"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle, bit for bit, on seeded scenes."""
from pathlib import Path

import numpy as np
import pytest

from garden_b200 import scenes, views as V
from garden_b200.layout import RT_COLOR, RT_OIT, RT_OPAQUE, RT_TRANSLUCENT, RT_UI, make_views

from common import OracleRun, aos_inputs, compare_gpu_to_oracle

pytestmark = pytest.mark.gpu


def _run_both(scene, views, strides=None, ready=None, draw_ready=None):
    from garden_b200.binding import ScenePrep
    t, pools = aos_inputs(scene, strides)
    rts = [p.render_type for p in scene.pools]
    orun = OracleRun((t, t.dtype.itemsize, t.size), [(m, m.dtype.itemsize, m.size) for m in pools], rts, views,
                     scene.camera_pos, ready=ready, draw_ready=draw_ready)
    sp = ScenePrep(0)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, rts[k], m, m.dtype.itemsize, m.size, m.size,
                         True if draw_ready is None else draw_ready[k], None if ready is None else ready[k])
    sp.set_views(views, scene.camera_pos)
    sp.run()
    compare_gpu_to_oracle(sp, orun, rts, views, scene.name)
    return sp, orun, t, pools


def test_c1_flat_single_view(oracle_built, sceneprep_lib):
    scene = scenes.config_scene("C1")
    views, _ = V.perspective_views([(0.4, -0.05)], 1.2, 16 / 9, 0.01)
    sp, orun, _, _ = _run_both(scene, views)
    assert orun.views[0]["unsorted"][0][1] > 500  # the frustum sees a real share of the scene


def test_depth4_camera_and_cascades(oracle_built, sceneprep_lib):
    scene = scenes.config_scene("C2", n=200_000)
    scene.camera_pos = np.array([5.0, 2.0, -3.0], np.float32)
    views, _ = V.camera_and_cascades(0.3, -0.1, 1.2, 16 / 9, 0.01, 100.0, (0.05, 0.1, 0.25, 1.0))
    _run_both(scene, views)


def test_depth8_opaque_and_translucent(oracle_built, sceneprep_lib):
    scene = scenes.config_scene("C3", n=150_000)
    views, _ = V.perspective_views([(1.1, 0.05)], 1.3, 16 / 9, 0.01)
    _run_both(scene, views, strides=[48, 64])


# ---- every branch of the filters and buckets (tests/edge_scenes.py) -------------------------------------------------
def test_mixed_scene_all_branches(oracle_built, sceneprep_lib):
    from edge_scenes import mixed_scene, mixed_views
    scene = mixed_scene(seed=21, n=60_000, box_half=120.0)
    views = mixed_views(yaw=1.3)
    ready = [p.ready for p in scene.pools]
    sp, orun, t, pools = _run_both(scene, views, ready=ready)
    main = orun.views[-1]
    assert main["ui"][1] > 0 and main["trans"][1] > 0
    # isVisible write-back (main view only, mesh.cpp:144-146,152-153,161-167) against the oracle's per-slot result
    for k, m in enumerate(pools):
        raw = m.view(np.uint8).reshape(-1, m.dtype.itemsize)
        raw[:, 15] = 0xFF
        sp.writeback_visible(k, m, m.dtype.itemsize)
        want = main["visible"][k]
        assert np.array_equal(raw[:, 15], want), f"pool {k}: isVisible differs"
    sp.close()


def test_few_planes_and_freed_slots(oracle_built, sceneprep_lib):
    from edge_scenes import few_planes_views, mixed_scene
    scene = mixed_scene(seed=22, n=20_000, with_ui=False, box_half=80.0)
    t, pools = aos_inputs(scene)
    # free slots: default-constructed components (entity == 0) in the middle of the pools (linear-pool.hpp)
    leaves = np.ones(scene.entity_count, bool)
    leaves[scene.parent[scene.parent >= 0]] = False
    dead = set((np.nonzero(leaves)[0][::5] + 1).tolist())
    for arr in [t] + pools:
        kill = np.isin(arr["entity"], list(dead))
        raw = arr.view(np.uint8).reshape(-1, arr.dtype.itemsize)
        raw[kill] = 0
    from garden_b200.binding import ScenePrep
    views = few_planes_views()
    rts = [p.render_type for p in scene.pools]
    ready = [p.ready for p in scene.pools]
    orun = OracleRun((t, t.dtype.itemsize, t.size), [(m, m.dtype.itemsize, m.size) for m in pools], rts, views,
                     scene.camera_pos, ready=ready)
    sp = ScenePrep(0)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, rts[k], m, m.dtype.itemsize, m.size, m.size, True, ready[k])
    sp.set_views(views, scene.camera_pos)
    sp.run()
    compare_gpu_to_oracle(sp, orun, rts, views, "freed")
    sp.close()


def test_dirty_range_updates_and_view_changes(oracle_built, sceneprep_lib):
    """C3's animated 10% (gsp_update_transforms on dirty ranges) over several frames, the camera moving each frame."""
    from garden_b200.binding import ScenePrep
    scene = scenes.config_scene("C3", n=50_000)
    t, pools = aos_inputs(scene, strides=[48, 64])
    rts = [p.render_type for p in scene.pools]
    sp = ScenePrep(0)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, rts[k], m, m.dtype.itemsize, m.size)
    for frame in range(3):
        sel, p, r, s = scenes.animate_trs(scene, frame, 99)
        t["position"][sel] = p; t["rotation"][sel] = r; t["scale"][sel] = s
        # the caller knows its dirty set; here: one range per run of 4096 slots that contains an animated slot
        for first in range(0, t.size, 4096):
            sp.update_transforms(t, t.dtype.itemsize, first, min(4096, t.size - first))
        cam = np.array([1.0 + frame, 0.5, -2.0 * frame], np.float32)
        views, _ = V.perspective_views([(0.2 + 0.4 * frame, 0.0)], 1.3, 16 / 9, 0.01)
        sp.set_views(views, cam)
        sp.run()
        orun = OracleRun((t, t.dtype.itemsize, t.size), [(m, m.dtype.itemsize, m.size) for m in pools], rts, views, cam)
        compare_gpu_to_oracle(sp, orun, rts, views, f"frame {frame}")
    sp.close()


def test_indexed_updates_match_full_restage(oracle_built, sceneprep_lib):
    """C3's animated tenth as a SCATTERED dirty set (gsp_update_transforms_indexed): only the listed components travel; the
    frame equals the oracle on the fully updated pool. Also: duplicates in the list, an out-of-range slot."""
    from garden_b200.binding import ScenePrep, ScenePrepError
    scene = scenes.config_scene("C3", n=60_000)
    t, pools = aos_inputs(scene, strides=[64, 48])
    rts = [p.render_type for p in scene.pools]
    sp = ScenePrep(0)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, rts[k], m, m.dtype.itemsize, m.size)
    for frame in range(3):
        sel, p, r, s = scenes.animate_trs(scene, frame, 41)
        t["position"][sel] = p; t["rotation"][sel] = r; t["scale"][sel] = s
        slots = sel if frame != 1 else np.concatenate([sel, sel[:100]])  # (entity index == transform slot in this scene)
        sp.update_transforms_indexed(t, t.dtype.itemsize, slots)
        cam = np.array([1.0 + frame, 0.5, -2.0 * frame], np.float32)
        views, _ = V.perspective_views([(0.2 + 0.4 * frame, 0.0)], 1.3, 16 / 9, 0.01)
        sp.set_views(views, cam)
        sp.run()
        orun = OracleRun((t, t.dtype.itemsize, t.size), [(m, m.dtype.itemsize, m.size) for m in pools], rts, views, cam)
        compare_gpu_to_oracle(sp, orun, rts, views, f"indexed frame {frame}")
    with pytest.raises(ScenePrepError):
        sp.update_transforms_indexed(t, t.dtype.itemsize, np.array([t.size], np.uint32))
    sp.close()


def test_world_matrices_within_2ulp(oracle_built, sceneprep_lib):
    """north_star: world matrices within 2 ulp of the reference's calcModel — they are in fact bit-identical."""
    import reflib
    from garden_b200.binding import ScenePrep
    scene = scenes.config_scene("C4", n=30_000)
    scene.camera_pos = np.array([12.5, 3.0, -7.25], np.float32)
    views, _ = V.perspective_views([(0.0, 0.0), (3.14, 0.0), (1.57, 0.0), (-1.57, 0.0)], 1.6, 1.0, 0.01)
    t, pools = aos_inputs(scene)
    sp = ScenePrep(0)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(1)
    sp.set_mesh_pool(0, RT_OPAQUE, pools[0], 48, pools[0].size)
    sp.set_views(views, scene.camera_pos)
    sp.run()
    models = sp.download_models(0, pools[0].size)
    vis = np.zeros(pools[0].size, bool)
    for v in range(views.size):
        rec, _, _ = sp.get_unsorted(v, 0)
        vis[(rec["componentOffset"] // 48).astype(np.int64)] = True
    assert vis.sum() > 5000
    o = reflib.Oracle()
    o.set_transforms(t, t.dtype.itemsize, t.size)
    worst = 0
    for slot in np.nonzero(vis)[0][::7]:
        want = o.calc_model(int(slot), scene.camera_pos).reshape(4, 4)[:, :3].reshape(12)
        a, b = models[slot].view(np.int32).astype(np.int64), want.view(np.int32).astype(np.int64)
        worst = max(worst, int(np.abs(a - b).max()))
    assert worst <= 2, f"world matrices differ by {worst} ulp"
    assert worst == 0
    sp.close()


# ---- error behaviour of the boundary (the reference throws EcsmError / GardenError; here: status codes) -------------------
def test_errors_are_status_codes(sceneprep_lib):
    from garden_b200.binding import GSP_ERR_HIERARCHY, GSP_ERR_INVALID, GSP_ERR_STATE, ScenePrep, ScenePrepError
    scene = scenes.config_scene("C2", n=1000)
    t, pools = aos_inputs(scene)
    sp = ScenePrep(0)
    with pytest.raises(ScenePrepError) as e:
        sp.run()  # no views yet
    assert e.value.code == GSP_ERR_STATE
    with pytest.raises(ScenePrepError) as e:
        sp.set_transforms(t, 72, t.size)  # stride smaller than sizeof(TransformComponent)
    assert e.value.code == GSP_ERR_INVALID
    bad = t.copy()
    bad["parent"][10] = 5_000_000  # parent entity without a TransformComponent: Manager::get throws (ecsm.hpp:863-873)
    with pytest.raises(ScenePrepError) as e:
        sp.set_transforms(bad, bad.dtype.itemsize, bad.size)
    assert e.value.code == GSP_ERR_HIERARCHY
    cyc = t.copy()
    cyc["parent"][0] = cyc["entity"][4]  # 0 -> 4 -> 3 -> 2 -> 1 -> 0
    sp.set_transforms(cyc, cyc.dtype.itemsize, cyc.size)
    sp.set_pool_count(1)
    sp.set_mesh_pool(0, RT_OPAQUE, pools[0], 48, pools[0].size)
    views, _ = V.perspective_views([(0.0, 0.0)], 1.2, 1.0, 0.01)
    sp.set_views(views, np.zeros(3, np.float32))
    with pytest.raises(ScenePrepError) as e:
        sp.run()
    assert e.value.code == GSP_ERR_HIERARCHY
    with pytest.raises(ScenePrepError):
        sp.get_unsorted(0, 0)  # no completed frame
    sp.close()


def test_empty_inputs(sceneprep_lib):
    from garden_b200.binding import ScenePrep
    sp = ScenePrep(0)
    t = np.zeros(0, dtype=np.dtype([("x", "u1", 80)]))
    sp.set_transforms(None, 80, 0)
    sp.set_pool_count(2)
    sp.set_mesh_pool(0, RT_OPAQUE, None, 48, 0)
    sp.set_mesh_pool(1, RT_TRANSLUCENT, None, 48, 0)
    views, _ = V.perspective_views([(0.0, 0.0)], 1.2, 1.0, 0.01)
    sp.set_views(views, np.zeros(3, np.float32))
    sp.run()
    assert sp.unsorted_buffer_count(0) == 1 and sp.sorted_buffer_count(0) == 1
    rec, draw, inst = sp.get_unsorted(0, 0)
    assert (rec.size, draw, inst) == (0, 0, 0)
    assert sp.get_sorted(0, 0)[1] == 0 and sp.last_visible_total() == 0
    sp.close()


# ---- full BASELINE sizes: EVERY list of EVERY view against the reference build ----------------------------------------
FULL_SIZE = [("C2", 1_000_000), ("C3", 4_000_000), ("C4", 16_000_000)]
FULL_SIZE_SAMPLES = Path(__file__).resolve().parent / "golden" / "full_size" / "samples.npz"
SAMPLE_ROWS = 128


def _full_size_inputs(scene):
    """(transform bytes, stride, occupancy, [(pool bytes, stride, occupancy, count)]) of scenes.build_aos(scene)."""
    tt, pp = scenes.build_aos(scene)
    pools = [(m.view(np.uint8).reshape(m.size, m.dtype.itemsize), m.dtype.itemsize, m.size, m.size) for m in pp]
    return tt.view(np.uint8).reshape(tt.size, 80), 80, tt.size, pools


def full_size_sample(frames, workload: str) -> dict:
    """A fixed sample of OracleRun-shaped results: per list its counts, and the raw 64 bytes (key bits, slot, bakedModel
    bits, buffer index) of SAMPLE_ROWS seeded row positions, which pin the draw order there."""
    out = {}
    for v, f in enumerate(frames):
        lists = [(f"unsorted{b}", rec, draw, inst) for b, (rec, draw, inst) in enumerate(f["unsorted"])]
        lists += [("trans", *f["trans"], 0), ("ui", *f["ui"], 0)]
        out[f"{workload}_v{v}_sorted_counts"] = np.array(f["sorted_counts"], np.int64).reshape(-1, 2)
        for i, (name, rec, draw, inst) in enumerate(lists):
            rows = np.arange(draw)
            if draw > SAMPLE_ROWS:
                rows = np.sort(np.random.default_rng([v, i]).choice(draw, SAMPLE_ROWS, replace=False))
            out[f"{workload}_v{v}_{name}_counts"] = np.array([draw, inst], np.int64)
            out[f"{workload}_v{v}_{name}_rows"] = rows.astype(np.int64)
            out[f"{workload}_v{v}_{name}_records"] = np.ascontiguousarray(rec[:draw][rows]).view(np.uint8).reshape(-1, 64)
    return out


def make_full_size_samples():
    """Writes FULL_SIZE_SAMPLES from the oracle's results on the inputs test_full_size_vs_reference uses without oracle/_ref
    (CPU only, a few minutes): `PYTHONPATH=.:tests python -c "import test_gpu_parity as t; t.make_full_size_samples()"`."""
    import bench
    out = {}
    for workload, n in FULL_SIZE:
        scene = scenes.config_scene(workload, n=n)
        scene.camera_pos = bench.camera_pos()
        views = bench.frame_views(workload)
        t, tstride, tocc, pools = _full_size_inputs(scene)
        rts = [p.render_type for p in scene.pools]
        frames = OracleRun((t, tstride, tocc), [(p[0], p[1], p[2]) for p in pools], rts, views, scene.camera_pos).views
        out.update(full_size_sample(frames, workload))
    np.savez_compressed(FULL_SIZE_SAMPLES, **out)
    print(f"{FULL_SIZE_SAMPLES}: {FULL_SIZE_SAMPLES.stat().st_size / 1024:.0f} KiB")


@pytest.mark.parametrize("workload,n", FULL_SIZE)
def test_full_size_vs_reference(sceneprep_lib, oracle_built, workload, n):
    """At BASELINE.json's sizes: the scene is built through the reference's real ECS (oracle/_ref parity build: the
    reference's own mesh.cpp / transform.cpp, SURVEY.md 8c), the CUDA path consumes the raw bytes of the reference's live
    pools, and every draw list of every view is compared with the reference's — key bits, draw order (the reference's
    order canonicalised inside equal-key runs, ours must already be canonical), bakedModel bits, counts — plus isVisible of
    every slot. A wrongly culled entity anywhere in the scene fails this test. Without oracle/_ref (a clean checkout) the
    pinned C oracle takes the reference's place, and a stored sample of the lists (tests/golden/full_size/samples.npz, see
    full_size_sample) must match as well, so that a change made alike to the oracle and the CUDA path is still caught. Then
    idempotence: a second frame over the same state gives identical lists."""
    import bench
    import reflib
    from common import assert_frames_equal, gpu_frame, ref_frame
    from garden_b200.binding import ScenePrep
    scene = scenes.config_scene(workload, n=n)
    scene.camera_pos = bench.camera_pos()
    views = bench.frame_views(workload)
    rts = [p.render_type for p in scene.pools]
    if reflib.ref_available("parity"):
        ref = reflib.RefEngine("parity", threads=-1)
        ref.load_scene(scene)
        _, tstride, tocc = ref.transform_pool()
        t = ref.transform_bytes().reshape(tocc, tstride).copy()
        pools = []
        for k in range(len(rts)):
            _, stride, occ, cnt = ref.mesh_pool(k)
            pools.append((ref.pool_bytes(k).reshape(occ, stride).copy(), stride, occ, cnt))
        want = ref_frame(ref, views)
        ref.close()
        canonicalise_want = True
    else:
        t, tstride, tocc, pools = _full_size_inputs(scene)
        want = OracleRun((t, tstride, tocc), [(p[0], p[1], p[2]) for p in pools], rts, views, scene.camera_pos).views
        stored = np.load(FULL_SIZE_SAMPLES)
        got_sample = full_size_sample(want, workload)
        assert sorted(got_sample) == sorted(k for k in stored.files if k.startswith(workload + "_"))
        for k, a in got_sample.items():
            assert np.array_equal(a, stored[k]), f"{workload} {n}: {k} differs from the stored sample"
    del scene
    sp = ScenePrep(0)
    sp.set_transforms(t, tstride, tocc)
    sp.set_pool_count(len(pools))
    for k, (raw, stride, occ, cnt) in enumerate(pools):
        sp.set_mesh_pool(k, rts[k], raw, stride, occ, cnt)
    sp.set_views(views, bench.camera_pos())
    sp.run()
    got = gpu_frame(sp, views, [(p[0], p[1]) for p in pools])
    total = sum(u[1] for f in got for u in f["unsorted"]) + sum(f["trans"][1] for f in got)
    assert total == sp.last_visible_total() and total > n // 50
    assert_frames_equal(got, want, rts, f"{workload} {n}", canonicalise_got=False)
    del want
    # idempotence: a second frame over the same state gives identical lists
    sp.run()
    again = gpu_frame(sp, views)
    for v, (a, b) in enumerate(zip(got, again)):
        for (ra, da, ia), (rb, db, ib) in zip(a["unsorted"], b["unsorted"]):
            assert (da, ia) == (db, ib) and np.array_equal(ra, rb), f"view {v}: second frame differs"
        assert a["trans"][1] == b["trans"][1] and np.array_equal(a["trans"][0], b["trans"][0])
    sp.close()


def test_exact_arithmetic_shortcuts_on_device(sceneprep_lib):
    """The hot kernel's cheaper instruction sequences (shared-reciprocal division, sqrt fast path, folded products, packed
    FP32 pairs) against the reference's 4-lane IEEE operation order, bit for bit, over ~1.2e9 random / adversarial inputs."""
    from garden_b200.binding import load_library
    lib = load_library()
    res = np.zeros(5, dtype=np.uint64)
    for seed in (1, 2):
        rc = lib.gsp_selftest_math(0, 148 * 8, 2048, seed, res.ctypes.data)
        assert rc == 0
        tested, fast, bad, mm_tested, mm_bad = (int(x) for x in res)
        assert tested == 148 * 8 * 256 * 2048
        assert fast > tested * 0.6 and mm_tested > tested * 0.4, (tested, fast, mm_tested)
        print(f"selftest seed {seed}: tested {tested}, shortcut taken {fast}, mismatches {bad}; products {mm_tested}, mismatches {mm_bad}")
        assert bad == 0, f"{bad} of {fast} shortcut results differ from the exact code"
        assert mm_bad == 0, f"{mm_bad} of {mm_tested} packed products differ"
