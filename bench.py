#!/usr/bin/env python
"""Benchmark of the scene-preparation hot path (transform -> cull -> key -> compact -> sort -> draw records).

  python bench.py --gpus N --steps K --warmup W                 the B200 path (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K --warmup W   the reference's own CPU thread-pool path

One JSON line on stdout (rank 0). A "step" is one frame = all views of one scene state; exactly --steps frames are timed.
Metric: entities transformed+culled+sorted per second (BASELINE.json). `value` is device-resident (SoA already in HBM, lists
left in HBM), `e2e` goes through the C ABI with host buffers (AoS upload, list download, isVisible write-back) every step.
--dump-outputs DIR writes the draw lists of the last timed step (same arguments, same seeded inputs, same files).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
_JSON_OUT = sys.stdout

from garden_b200 import scenes, views as V  # noqa: E402

METRIC = "entities transformed+culled+sorted/s"
UNIT = "entities/s"
# SURVEY.md §8d: algorithmic bytes per frame B = 75*N + 132*SumVis
BYTES_PER_ENTITY = 75
BYTES_PER_VISIBLE = 132
WORKLOADS = {
    # name -> (config, default N, description)
    "C4": ("C4", 16_000_000, "16M instances, depth-8 hierarchy, camera + 4 CSM cascades"),
    "C2": ("C2", 1_000_000, "1M entities, depth-4 hierarchy, camera + 4 CSM cascades"),
    "C3": ("C3", 4_000_000, "4M entities, depth-8, opaque + translucent, 1 view"),
    # configs[4]: 64M entities over 8 GPUs = 8M per GPU (weak-scaling shard), 16 independent views
    "C5": ("C5", 8_000_000, "64M entities / 8 GPUs (8M per GPU), depth-8, 16 independent views (2 cube probes + 4 split-screen)"),
}
SHADOW_DISTANCE = 100.0  # csm.hpp:88 default; --shadow-distance raises it so that the cascades see a larger share of the scene
CUBE_FACES = [(0.0, 0.0), (1.5707964, 0.0), (3.1415927, 0.0), (-1.5707964, 0.0), (0.0, 1.5), (0.0, -1.5)]  # (yaw, pitch)


def frame_views_vps(workload: str):
    """(views, viewProj matrices) of one frame of the workload."""
    if workload == "C3":
        return V.perspective_views([(0.6, -0.05)], 1.2, 16 / 9, 0.01)
    if workload == "C5":
        # two cube-map probes (6 faces each, 90 degree fov, aspect 1; the second rotated by 0.4 rad) + 4 split-screen cameras
        a, va = V.perspective_views(CUBE_FACES, 1.5707964, 1.0, 0.01)
        b, vb = V.perspective_views([(y + 0.4, p * 0.9) for y, p in CUBE_FACES], 1.5707964, 1.0, 0.01)
        c, vc = V.perspective_views([(0.3, -0.1), (1.9, -0.05), (3.6, -0.12), (5.1, -0.08)], 1.2, 16 / 9, 0.01)
        return np.concatenate([a, b, c]), list(va) + list(vb) + list(vc)
    return V.camera_and_cascades(0.6, -0.12, 1.2, 16 / 9, 0.01, SHADOW_DISTANCE, (0.05, 0.1, 0.25, 1.0))


def frame_views(workload: str):
    return frame_views_vps(workload)[0]


def camera_pos():
    return np.array([12.5, 3.0, -7.25], dtype=np.float32)


def load_traffic(workload: str, n: int, kernel_prefix: str):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of the same workload and
    size (profiles/*_ncu_traffic_*.json, written by tools/ncu_traffic.py); None when no capture matches."""
    for path in sorted((ROOT / "profiles").glob("*ncu_traffic*.json"), reverse=True):
        try:
            doc = json.loads(path.read_text())
        except Exception:
            continue
        if doc.get("workload") != workload or int(doc.get("entities", 0)) != n:
            continue
        # kernel_prefix may name several kernels ("kPrepass+kCompactSurvivors+kCull"): one launch of each, summed
        total, found = 0, 0
        for want in kernel_prefix.split("+"):
            for k in doc.get("kernels", []):
                if want in k["kernel"]:
                    total += int(k["traffic_bytes"]); found += 1
                    break
        if found == len(kernel_prefix.split("+")):
            return {"bytes": total, "source": f"profiles/{path.name}"}
    return None


def load_peaks():
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.rows = []
        self.proc = None
        self.device_index = device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.device_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first_sample(self, timeout: float = 5.0):
        t0 = time.time()
        while not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def stop(self, t_begin: float = 0.0, t_end: float = 1e300):
        """Summary of the samples whose arrival time lies inside [t_begin, t_end] (the timed region)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        inside = [row for t, row in self.rows if t_begin <= t <= t_end + 0.03]
        for row in inside:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm)}


def pinned_like(arr: np.ndarray):
    """Copies `arr` into pinned host memory (torch allocator) and returns (numpy view, owner tensor)."""
    import torch
    t = torch.empty(arr.nbytes, dtype=torch.uint8, pin_memory=True)
    view = t.numpy().view(arr.dtype).reshape(arr.shape)
    view[...] = arr
    return view, t


# ----------------------------------------------------------------------------------------------------------------------
REF_BUDGET_S = float(os.environ.get("GSP_REF_BUDGET_S", "240"))  # wall-clock bound of the reference arm's timed frames


def reference_engine_run(workload: str, sample_n: int, steps: int, warmup: int, seed: int):
    """Times the reference's own prepareMeshes (oracle/_ref stock build; falls back to the C port) on `sample_n`
    entities of the workload. Returns dict(value, ms_per_step, cores, kind, sample, visible)."""
    sys.path.insert(0, str(ROOT / "tests"))
    import reflib
    cfg = WORKLOADS[workload][0]
    scene = scenes.config_scene(cfg, n=sample_n, seed=seed)
    scene.camera_pos = camera_pos()
    views = frame_views(workload)
    if reflib.ref_available("stock"):
        ms = None
        while ms is None:
            with reflib.RefEngine("stock", threads=-1) as ref:
                ref.load_scene(scene)
                threads = ref.thread_count
                warm, _ = ref.time_frames(views, max(warmup, 1))
                # EXACTLY `steps` timed frames; if that many frames of the whole workload would not end within a few
                # minutes (REF_BUDGET_S), every step runs on a smaller scene of the same generator instead (the metric
                # is per entity). One retry at most: the second scene is sized from the first one's measured frame time.
                need_s = float(np.min(warm)) * 1e-3 * steps
                if need_s > REF_BUDGET_S and sample_n > 200_000:
                    chain = scenes.CONFIGS[cfg]["depth"] + 1
                    sample_n = max(int(sample_n * REF_BUDGET_S / need_s), 200_000) // chain * chain
                    scene = scenes.config_scene(cfg, n=sample_n, seed=seed)
                    scene.camera_pos = camera_pos()
                    continue
                ms, vis = ref.time_frames(views, steps)
        kind = "reference"
        cores = threads
    else:
        from common import OracleRun, aos_inputs
        t, pools = aos_inputs(scene)
        rts = [p.render_type for p in scene.pools]
        ms = []
        vis = [0]
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            orun = OracleRun((t, t.dtype.itemsize, t.size), [(m, m.dtype.itemsize, m.size) for m in pools], rts, views,
                             scene.camera_pos)
            if i >= warmup:
                ms.append((time.perf_counter() - t0) * 1e3)
            vis = [sum(u[1] for vw in orun.views for u in vw["unsorted"]) + sum(vw["trans"][1] for vw in orun.views)]
        ms = np.array(ms)
        kind, cores = "port", 1
    mean_ms = float(np.mean(ms))
    return {"value": sample_n / (mean_ms * 1e-3), "ms_per_step": mean_ms, "best_ms": float(np.min(ms)), "cores": int(cores),
            "kind": kind, "visible": int(vis[-1]), "entities": int(sample_n),
            "sample": f"{sample_n} entities of workload {workload} (same generator, same {views.size} views), "
                      f"{len(ms)} frames, mean"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    whole = WORKLOADS[args.workload][1]
    res = reference_engine_run(args.workload, args.ref_sample or whole, args.steps, args.warmup, args.seed)
    sample = res["entities"]
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload][2]}", "entities_per_gpu": sample,
                   "entities_total": sample, "entities_per_step": sample,
                   "views": int(frame_views(args.workload).size), "visible_total": res["visible"],
                   "same_config": sample == whole,
                   "note": ("the reference's own prepareMeshes (thread pool on all host cores) over "
                            + ("the WHOLE workload" if sample == whole else f"a {sample}-entity sample of the workload (time budget {REF_BUDGET_S:.0f} s for {args.steps} steps)")
                            + ", one call per view per step as mesh.cpp:795-847,893-903 does")},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_JSON_OUT, flush=True)



# ----------------------------------------------------------------------------------------------------------------------
def shard_scene(whole, a: int, b: int):
    """Entities [a, b) of `whole` as a scene of their own (a and b at hierarchy boundaries: parents stay inside)."""
    pools = []
    for pd in whole.pools:
        sel = (pd.entity_index >= a) & (pd.entity_index < b)
        pools.append(scenes.PoolDesc(pd.render_type, (pd.entity_index[sel] - a).astype(np.uint32), pd.aabb[sel],
                                     None if pd.enabled is None else pd.enabled[sel], None if pd.ready is None else pd.ready[sel],
                                     pd.stride, pd.draw_ready))
    return scenes.SceneDesc(whole.position[a:b], whole.rotation[a:b], whole.scale[a:b],
                            np.where(whole.parent[a:b] >= 0, whole.parent[a:b] - a, -1).astype(np.int32), whole.tflags[a:b],
                            pools, None, whole.camera_pos, whole.name)


def stage_scene(sp, scene, views):
    t, pools = scenes.build_aos(scene)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, scene.pools[k].render_type, m, m.dtype.itemsize, m.size)
    sp.set_views(views, scene.camera_pos)
    return [m.size for m in pools]


DUMP_BYTES = 64 << 20
RECORD_COLUMNS = 16  # row in the list, componentOffset, bakedModel[12], distanceSq, bufferIndex


def dump_outputs(sp, views, out_dir: Path, seed: int):
    """Writes what a caller of the frame receives (gsp_get_unsorted, gsp_get_sorted, gsp_get_sorted_counts) as float64 .npy
    files, so that two builds can be compared output for output:
      counts.npy    one row (view, list, buffer, drawCount, instanceCount) per list of every view: list 0 = unsorted buffer,
                    1 = translucent list, 2 = UI list (their instanceCount is 0: gsp_get_sorted returns none), 3 = sorted
                    buffer as gsp_get_sorted_counts reports it
      view<v>_unsorted<b>.npy, view<v>_translucent.npy, view<v>_ui.npy
                    rows of RECORD_COLUMNS, one per draw record, in list order; written for the non-empty lists only
    Every field is exact in float64. Lists that do not fit DUMP_BYTES together are cut to samples of rows (short lists stay
    whole, the long ones share the rest evenly) whose positions depend only on `seed`, the list's index and the list lengths."""
    out_dir.mkdir(parents=True, exist_ok=True)

    def fetch(v, which, b):  # (records, drawCount, instanceCount)
        if which == 0:
            return sp.get_unsorted(v, b, copy=False)
        return (*sp.get_sorted(v, which - 1, copy=False), 0)

    lists, counts = [], []
    for v in range(views.size):
        lists += [(f"view{v}_unsorted{b}", v, 0, b) for b in range(sp.unsorted_buffer_count(v))]
        lists += [(f"view{v}_translucent", v, 1, 0), (f"view{v}_ui", v, 2, 0)]
    for _, v, which, b in lists:
        counts.append((v, which, b, *fetch(v, which, b)[1:]))
    counts += [(v, 3, b, *sp.get_sorted_counts(v, b)) for v in range(views.size) for b in range(sp.sorted_buffer_count(v))]
    np.save(out_dir / "counts.npy", np.array(counts, np.float64))
    sizes = [c[3] for c in counts[:len(lists)]]
    caps, left = [0] * len(lists), (DUMP_BYTES - (1 << 20)) // (8 * RECORD_COLUMNS)
    for k, i in enumerate(sorted(range(len(lists)), key=lambda i: sizes[i])):
        caps[i] = min(sizes[i], left // (len(lists) - k))
        left -= caps[i]
    for i, (name, v, which, b) in enumerate(lists):
        rec = fetch(v, which, b)[0]
        if rec.size == 0:
            continue
        rows = np.arange(rec.size)
        if rec.size > caps[i]:
            rows = np.sort(np.random.default_rng([seed, i]).choice(rec.size, caps[i], replace=False))
        sel = rec[rows]
        out = np.empty((rows.size, RECORD_COLUMNS), np.float64)
        out[:, 0] = rows
        out[:, 1] = sel["componentOffset"]
        out[:, 2:14] = sel["bakedModel"]
        out[:, 14] = sel["distanceSq"]
        out[:, 15] = sel["bufferIndex"]
        np.save(out_dir / f"{name}.npy", out)


def verify_exchange(workload: str, rank: int, world: int, local_rank: int, stream, per_rank: int = 180_000):
    """Merged-order check over the REAL exchange (NCCL inside the library): a reduced scene of world x per_rank entities is
    cut into contiguous ranges, every rank prepares its range and exchanges, rank 0 also sorts the WHOLE scene on its own GPU;
    the concatenated slices of every list must equal that single-GPU sort — key bits and (global) slot order."""
    import torch
    import torch.distributed as dist
    from garden_b200.binding import ScenePrep
    from garden_b200.dist import PipelinedRunMerger
    cfg = WORKLOADS[workload][0]
    chain = scenes.CONFIGS[cfg]["depth"] + 1
    per_rank = (per_rank // chain) * chain
    whole = scenes.config_scene(cfg, n=per_rank * world, seed=4321)
    whole.camera_pos = camera_pos()
    views = frame_views(workload)
    sp = ScenePrep(local_rank)
    sp.set_stream(stream.cuda_stream)
    stage_scene(sp, shard_scene(whole, rank * per_rank, (rank + 1) * per_rank), views)
    pm = PipelinedRunMerger(sp)
    for _ in range(2):
        pm.frame()
    pm.finish()
    mine = pm.last_result()["slices"]
    everyone = [None] * world
    dist.all_gather_object(everyone, [(s[0], s[1], s[2], s[3]) for s in mine])
    sp.close()
    out = None
    if rank == 0:
        one = ScenePrep(local_rank)
        one.set_stream(stream.cuda_stream)
        pool_sizes = stage_scene(one, whole, views)
        one.run()
        counts = one.list_counts().astype(np.int64)
        total = int(counts.sum())
        k = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
        p = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
        one.export_runs(k.data_ptr(), p.data_ptr(), max(total, 1))
        one.sync()
        torch.cuda.synchronize()
        kk, pp = k[:total].cpu().numpy().view(np.uint32), p[:total].cpu().numpy().view(np.uint32)
        one.close()
        # slot of a shard-local payload in the whole scene: pool slots are handed out in entity order, so rank r's slots of
        # pool q start where the lower ranks' slots of that pool end
        shard_pool_sizes = np.zeros((world, len(pool_sizes)), np.int64)
        for r in range(world):
            for q, pd in enumerate(whole.pools):
                shard_pool_sizes[r, q] = int(((pd.entity_index >= r * per_rank) & (pd.entity_index < (r + 1) * per_rank)).sum())
        first_slot = np.zeros_like(shard_pool_sizes)
        first_slot[1:] = np.cumsum(shard_pool_sizes, axis=0)[:-1]
        off, elements, ok = 0, 0, True
        for l in range(counts.size):
            want_k, want_p = kk[off:off + counts[l]], pp[off:off + counts[l]]
            off += int(counts[l])
            got_k, got_p = [], []
            pos = 0
            for r in range(world):
                start, gk, gp, gr = everyone[r][l]
                ok = ok and start == pos
                pos += gk.size
                pool = (gp >> 28).astype(np.int64)
                slot = (gp & 0x0FFFFFFF).astype(np.int64) + first_slot[gr.astype(np.int64), pool]
                got_k.append(gk); got_p.append(((pool << 28) | slot).astype(np.uint32))
            got_k, got_p = np.concatenate(got_k), np.concatenate(got_p)
            ok = ok and got_k.size == want_k.size and np.array_equal(got_k, want_k) and np.array_equal(got_p, want_p)
            elements += int(want_k.size)
        out = {"ok": bool(ok), "entities": int(per_rank * world), "lists": int(counts.size), "merged_elements": elements,
               "protocol": "alltoall" if pm.all_to_all else "allgather",
               "what": "slices of all ranks (real NCCL, exchange inside the library) concatenated == one single-GPU sort of the "
                       "whole scene: key bits and slot order, every list"}
        if not ok:
            raise RuntimeError(f"multi-GPU merged order differs from the single-GPU sort: {out}")
    dist.barrier()
    return out


def strong_scaling_point(args, rank: int, world: int, local_rank: int, stream):
    """Device-resident frame time with the workload's N in TOTAL, split over the ranks (contiguous ranges of ONE scene)."""
    import torch
    import torch.distributed as dist
    from garden_b200.binding import ScenePrep
    from garden_b200.dist import PipelinedRunMerger
    cfg, default_n, _ = WORKLOADS[args.workload]
    total = args.entities or default_n
    if args.workload == "C5":
        total = (args.entities or default_n) * 8  # configs[4]: 64M in total
    chain = scenes.CONFIGS[cfg]["depth"] + 1
    per = (total // world // chain) * chain
    scene = scenes.config_scene(cfg, n=per, seed=args.seed + 7919 * rank)  # (same generator and density as the weak shards)
    scene.camera_pos = camera_pos()
    views = frame_views(args.workload)
    sp = ScenePrep(local_rank)
    sp.set_stream(stream.cuda_stream)
    stage_scene(sp, scene, views)
    pm = PipelinedRunMerger(sp)
    for _ in range(max(args.warmup, 3)):
        pm.frame()
    pm.finish()
    sp.sync()
    frames = args.steps
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(frames):
        pm.frame()
    pm.finish()
    e1.record(stream)
    sp.sync()
    dist.barrier(); torch.cuda.synchronize()
    stats = torch.tensor([e0.elapsed_time(e1), float(sp.last_visible_total())], dtype=torch.float64, device="cuda")
    mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    ms = float(mx[0]) / frames
    sp.close()
    return {"scaling": "strong", "entities_total": int(per * world), "entities_per_gpu": int(per), "ms_per_step": ms,
            "value": per * world / (ms * 1e-3), "unit": UNIT, "visible_total": int(sm[1]), "frames_timed": frames,
            "protocol": "alltoall" if pm.all_to_all else "allgather"}

# ----------------------------------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from garden_b200.binding import ScenePrep

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the scene-preparation path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    cfg, default_n, desc = WORKLOADS[args.workload]
    n = args.entities or default_n
    merge_check, strong = None, None
    if world > 1:
        pre_stream = torch.cuda.Stream()
        torch.cuda.set_stream(pre_stream)
        if not args.no_verify:
            merge_check = verify_exchange(args.workload, rank, world, local_rank, pre_stream)
        if args.scaling in ("strong", "both"):
            strong = strong_scaling_point(args, rank, world, local_rank, pre_stream)
    # weak scaling: every GPU owns an N-entity shard (contiguous entity range of a world-size * N scene)
    scene = scenes.config_scene(cfg, n=n, seed=args.seed + 7919 * rank)
    scene.camera_pos = camera_pos()
    views = frame_views(args.workload)
    t_np, pools_np = scenes.build_aos(scene)
    rts = [p.render_type for p in scene.pools]
    t_pin, _t_owner = pinned_like(t_np)
    pool_pins = [pinned_like(m) for m in pools_np]
    del t_np, pools_np

    # a dedicated non-default stream: the library enqueues on it and torch.cuda.Event records on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = ScenePrep(local_rank)
    sp.set_stream(stream.cuda_stream)

    def stage():
        sp.set_transforms(t_pin, t_pin.dtype.itemsize, t_pin.size)
        sp.set_pool_count(len(pool_pins))
        for k, (m, _) in enumerate(pool_pins):
            sp.set_mesh_pool(k, rts[k], m, m.dtype.itemsize, m.size)
        sp.set_views(views, scene.camera_pos)

    stage()
    merger = None
    if world > 1:
        # exchange without host synchronisation, overlapped with the next frame (garden_b200.dist.PipelinedRunMerger)
        from garden_b200.dist import PipelinedRunMerger
        merger = PipelinedRunMerger(sp, overlap=not args.no_overlap)

    def frame():
        if merger is None:
            sp.run_async()
            return
        merger.frame()
        if merger.poll():
            raise RuntimeError("exchange block overflowed on a static scene")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ----
    for _ in range(max(args.warmup, 3)):
        frame()
    if merger is not None:
        merger.finish()
    sp.sync()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample()
    frames_timed = args.steps
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    ev0.record(stream)
    for _ in range(frames_timed):
        frame()
    if merger is not None:
        merger.finish()  # the compute stream waits for the last exchanges; every frame's flags are checked clean
    ev1.record(stream)
    sp.sync()
    barrier()
    t_end = time.time()
    elapsed_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        dump_outputs(sp, views, Path(args.dump_outputs), args.seed)
    # latency of ONE frame with nothing overlapped (cull + sort + emit + export + all-gather + merge, serialised)
    latency_ms = None
    exchange_bytes = 0
    exchange_parts = None
    if merger is not None:
        lat_steps = max(3, min(args.steps, 10))
        barrier()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        merger.timing = []
        l0.record(stream)
        for _ in range(lat_steps):
            merger.frame()
            merger.finish()
        l1.record(stream)
        sp.sync()
        barrier()
        latency_ms = l0.elapsed_time(l1) / lat_steps
        exchange_parts = merger.timing_summary()
        merger.timing = None
        exchange_bytes = merger.bytes_received()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    launches_per_step = sp.last_launch_count() + (merger.launches_per_frame if merger else 0)
    visible_total = sp.last_visible_total()

    # ---- per-kernel-group timing (CUDA events on the same stream, inside the library) ----
    sp.set_profiling(True)
    phase = np.zeros(6)
    prof_steps = max(3, min(args.steps, 10))
    for _ in range(prof_steps):
        sp.run()
        phase += sp.phase_times()
    phase /= prof_steps
    sp.set_profiling(False)

    # ---- SURVEY.md 8f rows, timed alone with CUDA events on the same stream (not part of the headline frame) ----
    next_rows = []
    if world == 1:
        peak_gbs, _ = load_peaks()
        # f1: instance data (mvp) of the main view's first buffer, straight into device memory
        vi = int(views.size) - 1  # the main camera is the last view of the frame (cascades first)
        _, main_draw, _ = sp.get_unsorted_device(vi, 0)
        if main_draw:
            inst = torch.empty(main_draw * 16, dtype=torch.float32, device="cuda")
            vp0 = np.asarray(frame_views_vps(args.workload)[1][vi], dtype=np.float32).reshape(16)
            sp.run_async()
            for _ in range(3):
                sp.emit_instances_device(vi, 0, 0, vp0, inst.data_ptr(), main_draw)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            a.record(stream)
            for _ in range(reps):
                sp.emit_instances_device(vi, 0, 0, vp0, inst.data_ptr(), main_draw)
            b.record(stream)
            sp.sync()
            ms = a.elapsed_time(b) / reps
            nbytes = main_draw * (48 + 64)  # bakedModel read + mvp write per instance
            next_rows.append({"row": "f1 instance mvp (kInstances)", "instances": int(main_draw), "ms": round(ms, 4),
                              "bytes": int(nbytes), "GBps": round(nbytes / (ms * 1e-3) / 1e9, 1),
                              "frac": round(nbytes / (ms * 1e-3) / 1e9 / peak_gbs, 3),
                              "note": "main-camera list; the record arena was just written, so part of the reads are L2 hits"})
            del inst
        # f3: setActive of 10k entities (deactivate, then reactivate: the scene is unchanged afterwards)
        ids = np.arange(1, min(n, 10_000 * 9) + 1, 9, dtype=np.uint32)  # chain roots of the generator's depth-8 chains
        t0 = time.perf_counter()
        sp.set_active(ids, False)
        t1 = time.perf_counter()
        sp.set_active(ids, True)
        t2 = time.perf_counter()
        nbytes = n * (2 + 2 + 4)  # flags read + written, parent link, per transform (ancestor re-reads hit L2)
        ms = min(t1 - t0, t2 - t1) * 1e3
        next_rows.append({"row": "f3 setActive (kSetSelfActive + kPropagateActive), host-timed incl. id upload + sync",
                          "entities_toggled": int(ids.size), "transforms": int(n), "ms": round(ms, 4), "bytes": int(nbytes),
                          "GBps": round(nbytes / (ms * 1e-3) / 1e9, 1), "frac": round(nbytes / (ms * 1e-3) / 1e9 / peak_gbs, 3)})

    # ---- end to end through the C ABI with host buffers ----
    # every step: the whole AoS pools + views go host -> device (the ECS has no dirty tracking; pinned memory is read in
    # place by the staging kernels), the frame runs, every draw list comes back, isVisible is stored into the host pool
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    records_bytes = 0
    parts = np.zeros(4)

    def e2e_frame(delta: bool = False):
        nonlocal records_bytes
        t0 = time.perf_counter()
        stage()
        t1 = time.perf_counter()
        sp.run()
        t2 = time.perf_counter()
        sp.fetch_all_async()  # the lists travel on the copy stream while isVisible is stored into the host pool
        changed = 0
        for k, (m, _) in enumerate(pool_pins):
            if delta:
                changed += sp.writeback_visible_delta(k, m, m.dtype.itemsize)
            else:
                sp.writeback_visible(k, m, m.dtype.itemsize)
        t3 = time.perf_counter()
        total = 0
        for v in range(views.size):
            for b in range(sp.unsorted_buffer_count(v)):
                rec, draw, _ = sp.get_unsorted(v, b, copy=False)  # (the first getter waits for the transfer)
                total += draw
            rec, draw = sp.get_sorted(v, 0, copy=False)
            total += draw
        t4 = time.perf_counter()
        parts[:] += (t1 - t0, t2 - t1, t3 - t2, t4 - t3)
        records_bytes = total * 64
        return total, changed

    # isVisible travels as the list of slots whose value differs from the byte the host holds (the library knows
    # that byte: it was uploaded with the pool or written by the previous write-back) — gsp_writeback_visible_delta
    e2e_frame(delta=True)  # (allocates the changed-slot list once; the first frame stores every visible slot)
    barrier()
    parts[:] = 0
    t0 = time.perf_counter()
    changed_total = 0
    for _ in range(e2e_steps):
        changed_total += e2e_frame(delta=True)[1]
    torch.cuda.synchronize()
    e2e_serial_s = (time.perf_counter() - t0) / e2e_steps
    e2e_serial_parts = (parts / e2e_steps * 1e3).round(3).tolist()

    # headline: the same steps software-pipelined the way an engine runs them — while the draw lists of frame k travel to the
    # host (copy stream, PCIe down), the inputs of frame k+1 are uploaded (PCIe up); the list getters keep serving the
    # snapshot gsp_fetch_all_async took until the next gsp_run. Every step still uploads all its inputs, runs its frame and
    # reads all the lists of a frame on the host.
    def consume_lists():
        total = 0
        for v in range(views.size):
            for b in range(sp.unsorted_buffer_count(v)):
                total += sp.get_unsorted(v, b, copy=False)[1]
            total += sp.get_sorted(v, 0, copy=False)[1]
        return total

    def produce():
        sp.run()
        sp.fetch_all_async()
        changed = 0
        for k, (m, _) in enumerate(pool_pins):
            changed += sp.writeback_visible_delta(k, m, m.dtype.itemsize)
        return changed

    stage()
    produce()  # frame 0 is in flight when the clock starts; the last frame's lists are awaited before it stops
    barrier()
    parts[:] = 0
    changed_total = 0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ta = time.perf_counter()
        stage()
        tb = time.perf_counter()
        records_bytes = consume_lists() * 64
        tc = time.perf_counter()
        changed_total += produce()
        td = time.perf_counter()
        parts[:] += (tb - ta, td - tc, 0.0, tc - tb)
    consume_lists()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e_parts = (parts / e2e_steps * 1e3).round(3).tolist()
    h2d = t_pin.nbytes + sum(m.nbytes for m, _ in pool_pins) + views.nbytes
    d2h = records_bytes + 4 * (changed_total // e2e_steps + len(pool_pins))
    # variant: every isVisible byte of every pool is rewritten from a bit mask (gsp_writeback_visible)
    e2e_frame()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_frame()
    torch.cuda.synchronize()
    e2e_delta_s = (time.perf_counter() - t0) / e2e_steps

    # variant: steady state of an engine that knows its dirty set — only the transforms that changed travel up
    # (gsp_update_transforms_indexed: C3 animates every tenth transform per frame; C2/C4/C5 scenes are static), the views are
    # set, the frame runs, every draw list and the changed isVisible bytes come back. Rank 0 only, reported, not the headline.
    incremental = None
    if rank == 0:
        if args.workload == "C3":
            dirty = np.arange(0, t_pin.size, 10, dtype=np.uint32)
        else:
            dirty = np.zeros(0, np.uint32)

        def inc_frame():
            if dirty.size:
                sp.update_transforms_indexed(t_pin, t_pin.dtype.itemsize, dirty)
            sp.set_views(views, scene.camera_pos)
            sp.run()
            sp.fetch_all_async()
            for k, (m, _) in enumerate(pool_pins):
                sp.writeback_visible_delta(k, m, m.dtype.itemsize)
            for v in range(views.size):
                for b in range(sp.unsorted_buffer_count(v)):
                    sp.get_unsorted(v, b, copy=False)
                sp.get_sorted(v, 0, copy=False)

        inc_frame()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            inc_frame()
        torch.cuda.synchronize()
        inc_s = (time.perf_counter() - t0) / e2e_steps
        incremental = {"value": n / inc_s, "ms_per_step": inc_s * 1e3, "dirty_transforms_per_step": int(dirty.size),
                       "h2d_bytes_per_step": int(dirty.size * (t_pin.dtype.itemsize + 4) + views.nbytes),
                       "d2h_bytes_per_step": int(records_bytes),
                       "what": "only dirty transforms up (gsp_update_transforms_indexed), all draw lists + changed isVisible "
                               "bytes down; per GPU"}

    # ---- reduce over ranks: max time, summed work ----
    stats = torch.tensor([elapsed_ms, e2e_s, float(visible_total), e2e_delta_s, latency_ms or 0.0], dtype=torch.float64,
                         device="cuda")
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        elapsed_ms, e2e_s, visible_sum, e2e_delta_s = float(mx[0]), float(mx[1]), float(sm[2]), float(mx[3])
        latency_ms = float(mx[4])
    else:
        visible_sum = float(visible_total)
    ms_per_step = elapsed_ms / frames_timed
    total_entities = n * world
    value = total_entities / (ms_per_step * 1e-3)

    if rank == 0:
        peak, peak_src = load_peaks()
        alg_bytes = BYTES_PER_ENTITY * n + BYTES_PER_VISIBLE * visible_total  # per GPU
        # the cull stage = filter + conservative prepass (kPrepass) + survivor compaction (kCompactSurvivors) + world matrices
        # and exact culling of the survivors (kCull, or kPrepassT/kCull<world>/kClassify on the split path): together they
        # consume the 75 B/entity input stream of SURVEY.md 8d, so the stage is one roofline entry
        phase = phase.copy()
        cull_parts = {"prepass + survivor compaction (kPrepass, kCompactSurvivors)": round(float(phase[3]), 4),
                      "world matrices + exact culling of the survivors (kCull)": round(float(phase[1]), 4)}
        phase[1] += phase[3]; phase[3] = 0.0
        names = ["link", "cull stage: filter + prepass + survivor compaction + world matrices + culling (kPrepass, kCompactSurvivors, kCull)",
                 "compaction + keys + sort histograms (kScanChunks + kScatter)",
                 "(unused)", "sort passes (kSortPass x4)", "record emission (kEmit)"]
        # algorithmic bytes attributed to each kernel group; they add up to 75*N + 132*SumVis (SURVEY.md 8d):
        # inputs + isVisible | the 4 B/key histogram read of the formula (done on the fly here) | - |
        # 4 x (8 read + 8 write) | 64 B record write
        kernel_bytes = [0, 75 * n, 4 * visible_total, 0, 64 * visible_total, 64 * visible_total]
        frame_ms = float(phase.sum())
        kernels = []
        for i in (1, 2, 4, 5):
            ms = float(phase[i])
            gbs = kernel_bytes[i] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            kernels.append({"name": names[i], "ms": round(ms, 4), "share": round(ms / frame_ms, 3) if frame_ms else 0,
                            "bytes": int(kernel_bytes[i]), "GBps": round(gbs, 1), "frac": round(gbs / peak, 3)})
            if i == 1:
                kernels[-1]["parts_ms"] = cull_parts
        dom = max(range(len(kernels)), key=lambda i: kernels[i]["ms"])
        frame_gbs = alg_bytes / (ms_per_step * 1e-3) / 1e9
        roofline = {
            "bound": "hbm", "kernel": kernels[dom]["name"], "achieved": kernels[dom]["GBps"], "peak": peak, "unit": "GB/s",
            "frac": kernels[dom]["frac"], "traffic": None, "peak_source": peak_src,
            "algorithmic_bytes": int(kernels[dom]["bytes"]),
            "frame": {"algorithmic_bytes": int(alg_bytes), "achieved": round(frame_gbs, 1), "frac": round(frame_gbs / peak, 3),
                      "formula": "75*N + 132*SumVis (SURVEY.md 8d), per GPU, over the timed ms_per_step"},
            "kernels": kernels,
        }
        kernel_symbol = {1: "kPrepass+kCompactSurvivors+kCull", 2: "kScatter", 4: "kSortPass", 5: "kEmit"}[(1, 2, 4, 5)[dom]]
        traffic = load_traffic(args.workload, n, kernel_symbol)
        if traffic:
            roofline["traffic"] = traffic["bytes"]
            roofline["traffic_source"] = traffic["source"] + " (dram__bytes_read.sum + dram__bytes_write.sum, one launch of each kernel of the entry)"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "entities_per_gpu": n, "entities_total": total_entities,
                       "frames_timed": frames_timed,
                       "timing": f"{args.steps} frames back to back between two CUDA events; ms_per_step is their mean",
                       "views": int(views.size), "visible_total": int(visible_sum), "shadow_distance": SHADOW_DISTANCE,
                       "l2": "inputs larger than L2 (%.2f GB of SoA streams per frame vs 126 MB L2)" % (75 * n / 1e9),
                       "sharding": ("contiguous entity ranges per GPU, all views per GPU; sorted runs exchanged over NCCL by "
                                    "key range (fixed-capacity blocks, no host synchronisation) and k-way merged; "
                                    "frame k's exchange " + ("is serialised with" if args.no_overlap else "overlaps")
                                    + " frame k+1's cull") if world > 1 else "single GPU"},
            "roofline": roofline,
            "e2e": {"value": total_entities / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "what": "full AoS pool upload from pinned host memory (ECS has no dirty tracking; read in place by the "
                            "staging kernels) + run + all draw lists to host + the isVisible bytes that changed stored into "
                            "the host pool (gsp_writeback_visible_delta)",
                    "pipelining": "frame k's lists travel down while frame k+1's inputs travel up; one upload, one run, one "
                                  "full set of lists read on the host per step",
                    "parts_ms": {"upload+stage (previous lists travelling meanwhile)": e2e_parts[0],
                                 "run + isVisible delta write-back": e2e_parts[1],
                                 "wait_for_previous_lists": e2e_parts[3]},
                    "serial": {"value": total_entities / e2e_serial_s, "ms_per_step": e2e_serial_s * 1e3,
                               "what": "the same step with nothing overlapped across frames: upload, run, lists down, then the next",
                               "parts_ms": {"upload+stage": e2e_serial_parts[0], "run": e2e_serial_parts[1],
                                            "isVisible_writeback (lists travelling meanwhile)": e2e_serial_parts[2],
                                            "wait_for_lists": e2e_serial_parts[3]}},
                    "changed_slots_per_step": changed_total / e2e_steps,
                    "full_writeback": {"value": total_entities / e2e_delta_s, "ms_per_step": e2e_delta_s * 1e3,
                                       "what": "same, but every isVisible byte rewritten (gsp_writeback_visible)"},
                    "incremental": incremental},
            "gpu_launches": int(launches_per_step * frames_timed),
            "clocks": clocks,
        }
        if next_rows:
            line["next_rows"] = next_rows
        if world > 1:
            line["exchange"] = {"frame_latency_ms_serialised": latency_ms, "bytes_received_per_rank": exchange_bytes,
                                "protocol": "alltoall" if merger.all_to_all else "allgather",
                                "collectives_per_frame": 2 if merger.all_to_all else 1, "host_syncs_per_frame": 0,
                                "where": "inside libgarden_sceneprep.so (gsp_exchange_async, NCCL loaded by the library)",
                                "parts_rank0": exchange_parts}
            line["config"]["merge_check"] = merge_check
            if strong is not None:
                line["config"]["strong"] = strong
        if world == 1 and not args.no_cpu_baseline:
            res = reference_engine_run(args.workload, args.ref_sample or n, args.ref_steps, 1, args.seed)
            line["cpu_baseline"] = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"],
                                    "sample": res["sample"], "ms_per_step": res["ms_per_step"]}
        print(json.dumps(line), file=_JSON_OUT, flush=True)
    sp.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # stdout carries exactly ONE JSON line: anything a library prints there (e.g. NCCL's version banner) is sent to stderr
    global _JSON_OUT, SHADOW_DISTANCE
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--entities", type=int, default=0, help="override N per GPU (default: the workload's N)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--ref-sample", type=int, default=0, help="entities the CPU reference runs on (0 = the whole workload)")
    ap.add_argument("--ref-steps", type=int, default=5, help="frames of the in-line cpu_baseline leg")
    ap.add_argument("--scaling", default="both", choices=["weak", "strong", "both"],
                    help="N > 1: weak = the workload's N per GPU, strong = the workload's N in total; both = weak is the "
                         "headline value and the strong-scaling numbers go under config.strong")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: wait for every frame's exchange before the next frame")
    ap.add_argument("--no-verify", action="store_true", help="N>1: skip the merged-order check against a single-GPU sort")
    ap.add_argument("--shadow-distance", type=float, default=0.0,
                    help="CSM shadow distance of the camera + cascades workloads (default 100: the reference's); larger values "
                         "let every cascade see 10-15 %% of the scene (SURVEY.md 8d)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the draw lists of the last one to DIR/<name>.npy (see dump_outputs); "
                         "one GPU only: the merged lists of the multi-GPU path are not written")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs writes the lists of the single-GPU B200 path: use it with --impl b200 on one GPU")
    if args.shadow_distance > 0:
        SHADOW_DISTANCE = args.shadow_distance
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
