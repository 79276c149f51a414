"""Parity at the shapes the other suites never reach: ECS memory laid out the way a live ECS leaves it (transform rows in any
order, sparse entity ids, mesh rows out of entity order, freed slots), every view-count instantiation of the cull kernels
(3, 6, 7 -> 8, 8, 9 -> 16, 16), all eight mesh systems with sixteen views, very wide and very deep hierarchies, list
lengths at the sort / compaction tile boundaries, long equal-key runs and the keys +0, subnormal and +inf.

Every case is compared bit for bit with the oracle (tests/common.compare_gpu_to_oracle plus the main view's isVisible
bytes) and asserts that the edge it is named after was reached, on the oracle's lists or on the inputs, so later tuning of
a scene or a kernel cannot quietly stop exercising it. test_edges_reached_on_the_oracle and
test_relocation_keeps_the_oracle_lists run the same scenes without a GPU. NaN keys are left out: the reference's order
for them is unspecified."""
from __future__ import annotations

import types

import numpy as np
import pytest

from garden_b200 import scenes, views as V
from garden_b200.layout import RT_COLOR, RT_OIT, RT_OPAQUE, RT_REFRACTED, RT_TRANSLUCENT, RT_TRANS_DEPTH, RT_UI
from garden_b200.scenes import PoolDesc, SceneDesc

from common import compare_gpu_to_oracle
from edge_scenes import mixed_scene, mixed_views, random_forest
from reflib import Oracle

SORT_TILE = 4096          # keys per tile of the radix sort (sceneprep_internal.h: kSortTile)
CLOSURE_ENTRIES = 32      # closure entries of a 64-survivor tile of the fused kCull (cull.cu: kEntries - kWarpTile)
ALL_VIEWS = 0xFFFF


# ---- frames: ECS bytes + views, run through the oracle and through the C ABI ----------------------------------------------
class Frame:
    def __init__(self, name, t, pools, rts, views, cam, ready=None, masks=None):
        self.name, self.t, self.pools, self.rts, self.views = name, t, pools, rts, views
        self.cam = np.asarray(cam, np.float32)
        self.ready = ready if ready is not None else [None] * len(pools)
        self.masks = masks if masks is not None else [ALL_VIEWS] * len(pools)


def frame_of(scene: SceneDesc, views, name: str, masks=None) -> Frame:
    t, pools = scenes.build_aos(scene)
    return Frame(name, t, pools, [p.render_type for p in scene.pools], views, scene.camera_pos,
                 [p.ready for p in scene.pools], masks)


def oracle_frame(f: Frame):
    """The oracle's lists of every view (OracleRun.views shape). A pool takes part in view v iff bit v of its mask is set:
    isDrawReady() is asked once per view (mesh.cpp:426,482), so the oracle gets the view's bit as its readiness."""
    o = Oracle()
    o.set_transforms(f.t, f.t.dtype.itemsize, f.t.size)
    for k, m in enumerate(f.pools):
        o.set_pool(k, f.rts[k], m, m.dtype.itemsize, m.size, None, True, f.ready[k])
    o.set_pool_count(len(f.pools))
    o.set_camera(f.cam)
    out = []
    for v in range(f.views.size):
        for k in range(len(f.pools)):
            bit = bool((f.masks[k] >> v) & 1)
            o.set_pool_draw_ready(k, bit, bit)
        assert o.prepare(f.views[v]) == 0
        res = {"unsorted": [o.get_unsorted(b) for b in range(o.unsorted_buffer_count())],
               "sorted_counts": [o.get_sorted_counts(b) for b in range(o.sorted_buffer_count())],
               "trans": o.get_sorted(0), "ui": o.get_sorted(1)}
        if int(f.views[v]["shadowPass"]) < 0:
            res["visible"] = [o.get_visible(k) for k in range(len(f.pools))]
        out.append(res)
    o.close()
    return types.SimpleNamespace(views=out)


def stage(sp, f: Frame):
    sp.set_transforms(f.t, f.t.dtype.itemsize, f.t.size)
    sp.set_pool_count(len(f.pools))
    for k, m in enumerate(f.pools):
        sp.set_mesh_pool(k, f.rts[k], m, m.dtype.itemsize, m.size, ready_counts=f.ready[k])
        sp.set_pool_view_mask(k, f.masks[k])
    sp.set_views(f.views, f.cam)


def compare_frame(sp, f: Frame, orun, tag: str):
    """Every list of every view, then isVisible of the last main view (which wins, like repeated prepareMeshes calls)."""
    compare_gpu_to_oracle(sp, orun, f.rts, f.views, tag)
    main = [v for v in range(f.views.size) if int(f.views[v]["shadowPass"]) < 0]
    if not main:
        return
    for k, m in enumerate(f.pools):
        if m.size == 0:
            continue
        got = m.copy()
        raw = got.view(np.uint8).reshape(-1, m.dtype.itemsize)
        raw[:, 15] = 0xFF
        sp.writeback_visible(k, got, m.dtype.itemsize)
        want = orun.views[main[-1]]["visible"][k]
        sel = want != 0xFF
        assert np.array_equal(raw[sel, 15], want[sel]), f"{tag} pool {k}: isVisible differs"


def run_gpu(f: Frame, orun):
    from garden_b200.binding import ScenePrep
    sp = ScenePrep(0)
    try:
        stage(sp, f)
        sp.run()
        compare_frame(sp, f, orun, f.name)
    finally:
        sp.close()


# ---- list helpers for the edge assertions -------------------------------------------------------------------------------
def lists(orun):
    """(view, name, records) of every list of the frame."""
    for v, res in enumerate(orun.views):
        for b, (rec, _, _) in enumerate(res["unsorted"]):
            yield v, f"unsorted{b}", rec
        yield v, "trans", res["trans"][0]
        yield v, "ui", res["ui"][0]


def longest_equal_key_run(rec) -> int:
    if rec.size == 0:
        return 0
    k = rec["distanceSq"].view(np.uint32)
    cut = np.flatnonzero(np.diff(k) != 0)
    edges = np.concatenate([[-1], cut, [k.size - 1]])
    return int(np.diff(edges).max())


def all_keys(orun) -> np.ndarray:
    return np.concatenate([r["distanceSq"] for _, _, r in lists(orun)] + [np.zeros(0, np.float32)])


# ---- relocation: the same scene as another ECS would lay it out ----------------------------------------------------------
def relocate(f: Frame, seed: int, order: str = "random", freed: int = 0) -> tuple[Frame, np.ndarray]:
    """Returns (frame, id_map) with the same scene in other ECS memory: transform rows permuted at random or reversed (every
    child before its parent: build_aos puts parents first), entity ids mapped by a seeded bijection onto sparse ids up to
    4 * E (parents may get larger ids than their children), every mesh pool's rows permuted independently, and `freed` free
    slots (entity 0, stale bytes of another row, as LinearPool leaves them) spread over each pool. Rows carry their own
    entity and parent ids, so the bytes stay a valid ECS. id_map[old id] = new id (id_map[0] = 0)."""
    rng = np.random.default_rng(seed)
    e_max = int(max([int(f.t["entity"].max(initial=0))] + [int(m["entity"].max(initial=0)) for m in f.pools]))
    id_map = np.zeros(e_max + 1, np.uint32)
    id_map[1:] = rng.choice(np.arange(1, 4 * e_max + 1, dtype=np.uint32), e_max, replace=False)

    def scatter_rows(a, perm, extra=None):
        out = a[perm].copy()
        out["entity"] = id_map[out["entity"]]
        if "parent" in a.dtype.names:
            out["parent"] = id_map[out["parent"]]
        if freed and a.size:
            stale = out[rng.integers(0, out.size, freed)].copy()
            stale["entity"] = 0
            at = np.sort(rng.integers(0, out.size + 1, freed))
            out = np.insert(out, at, stale)
            if extra is not None:
                extra = np.insert(extra[perm], at, rng.integers(0, 4, freed).astype(np.uint8))
        elif extra is not None:
            extra = extra[perm]
        return out, extra

    n = f.t.size
    tperm = rng.permutation(n) if order == "random" else np.arange(n)[::-1]
    t, _ = scatter_rows(f.t, tperm)
    pools, ready = [], []
    for m, r in zip(f.pools, f.ready):
        p, r2 = scatter_rows(m, rng.permutation(m.size), r)
        pools.append(p)
        ready.append(r2)
    return Frame(f"{f.name} relocated ({order}, seed {seed})", t, pools, f.rts, f.views, f.cam, ready, f.masks), id_map


def relocation_edges(f: Frame):
    """(children stored before their parent, children whose parent has the larger id, mesh rows out of id order)."""
    slot_of = {int(e): i for i, e in enumerate(f.t["entity"]) if e}
    ent, par = f.t["entity"].astype(np.int64), f.t["parent"].astype(np.int64)
    kids = np.flatnonzero((ent != 0) & (par != 0))
    before = sum(1 for i in kids if i < slot_of[int(par[i])])
    larger = int(np.count_nonzero(par[kids] > ent[kids]))
    unordered = sum(int(np.count_nonzero(np.diff(m["entity"][m["entity"] != 0].astype(np.int64)) < 0)) for m in f.pools)
    return before, larger, unordered, kids.size


# ---- scene builders --------------------------------------------------------------------------------------------------
def unit_quats(rng, n) -> np.ndarray:
    q = rng.normal(size=(n, 4))
    return (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)


def scene_from(parent, pos, rot, pools, camera_pos=(0.0, 0.0, 0.0), scale=None, name="") -> SceneDesc:
    n = len(parent)
    scl = np.ones((n, 3), np.float32) if scale is None else scale
    return SceneDesc(np.asarray(pos, np.float32), np.asarray(rot, np.float32), scl, np.asarray(parent, np.int32),
                     np.full(n, 3, np.uint8), pools, None, np.asarray(camera_pos, np.float32), name=name)


def view_set(n: int, shape: str, yaw: float = 0.3):
    """`cascades`: N - 1 cascades of one light (one box group) + the camera; `independent`: N main views around the camera
    (the C5 shard's shape), the last one wins isVisible."""
    if shape == "cascades":
        splits = tuple(float(s) for s in np.geomspace(0.04, 1.0, n - 1))
        views, _ = V.camera_and_cascades(yaw, -0.1, 1.2, 16 / 9, 0.05, 70.0, splits)
    else:
        views, _ = V.perspective_views([(yaw + 2 * np.pi * i / n, 0.15 * np.sin(i)) for i in range(n)], 1.3, 16 / 9, 0.05)
    assert views.size == n
    return views


def case_mixed_relocated(seed: int, order: str) -> Frame:
    scene = mixed_scene(seed=seed, n=2500, max_depth=20, with_ui=True, with_ready=True, box_half=50.0)
    f = frame_of(scene, mixed_views(yaw=0.2 + 0.1 * seed), f"mixed{seed}")
    return relocate(f, seed, order, freed=40)[0]


def case_c3_relocated(order: str) -> Frame:
    scene = scenes.config_scene("C3", n=24_000, seed=77)     # depth-8 chains, a quarter of the meshes translucent
    views, _ = V.camera_and_cascades(0.8, -0.1, 1.2, 16 / 9, 0.05, 60.0, (0.1, 0.3, 1.0))
    return relocate(frame_of(scene, views, "C3"), 5, order, freed=64)[0]


def case_views(n: int, shape: str) -> Frame:
    scene = mixed_scene(seed=300 + n, n=2500, max_depth=10, with_ui=False, with_ready=True, box_half=55.0)
    views = view_set(n, shape)
    full = (1 << n) - 1
    if shape == "cascades":
        # pool 2 only in the camera view (bit n - 1), pool 3 only in the cascades, pool 4 in the upper half of the views
        masks = [full, full, 1 << (n - 1), full >> 1, full & ~((1 << (n // 2)) - 1)]
    else:
        masks = [full, full & ~(1 << (n // 2)), full & ~0x5, full & ~((1 << (n // 2)) - 1) | 1, full]
    return frame_of(scene, views, f"{n} views ({shape})", masks)


EIGHT_POOLS = [RT_OPAQUE, RT_COLOR, RT_OIT, RT_REFRACTED, RT_TRANS_DEPTH, RT_OPAQUE, RT_TRANSLUCENT, RT_TRANSLUCENT]


def case_eight_pools(sparse: bool) -> Frame:
    """8 mesh systems x 16 views: 6 unsorted lists + the shared translucent list per view. sparse: one empty pool, one pool
    left out of views 9..12 and one that only takes part in views 8..15."""
    seed, n = 41, 6000
    parent = random_forest(seed, n, 6)
    pos, rot, scl = scenes.random_trs(seed, n, (-45, -6, -45, 45, 6, 45), parent >= 0, local_extent=2.0,
                                      scale_range=(0.7, 1.3))
    which = (scenes.hash_u01(seed, 400, np.arange(n, dtype=np.uint64)) * 8).astype(np.int64)
    if sparse:
        which[which == 4] = 3
    pools = []
    for k, rt in enumerate(EIGHT_POOLS):
        sel = np.flatnonzero(which == k).astype(np.uint32)
        pools.append(PoolDesc(rt, sel, scenes.unit_aabb(sel.size), stride=48 + 16 * (k % 3)))
    scene = SceneDesc(pos, rot, scl, parent, np.full(n, 3, np.uint8), pools, None, np.array([1.0, 0.5, -1.0], np.float32))
    masks = [ALL_VIEWS] * 8
    if sparse:
        masks[1] = ALL_VIEWS & ~0x1E00
        masks[6] = 0xFF00
    return frame_of(scene, view_set(16, "independent", 0.1), f"8 pools x 16 views{' (sparse)' if sparse else ''}", masks)


def case_wide_root() -> Frame:
    """One root with 20000 children (and a grandchild under every 8th child)."""
    rng = np.random.default_rng(11)
    n_kids = 20_000
    parent = np.concatenate([[-1], np.zeros(n_kids, np.int32), 1 + np.arange(0, n_kids, 8)]).astype(np.int32)
    n = parent.size
    pos = rng.uniform(-12, 12, (n, 3)).astype(np.float32)
    pos[0] = (0.0, 0.0, 25.0)
    rot = unit_quats(rng, n)
    ent = np.arange(n, dtype=np.uint32)
    pools = [PoolDesc(RT_OPAQUE, ent[ent % 3 != 0], scenes.unit_aabb(int((ent % 3 != 0).sum()))),
             PoolDesc(RT_TRANSLUCENT, ent[ent % 3 == 0], scenes.unit_aabb(int((ent % 3 == 0).sum())))]
    views = view_set(4, "cascades", 0.0)
    return frame_of(scene_from(parent, pos, rot, pools, (0.5, 0.0, -3.0)), views, "one root, 20000 children")


def interleaved_chains(chains: int = 256, depth: int = 12, inner: str = "none"):
    """`chains` chains of `depth` nodes, stored level by level (node d of chain c at slot d * chains + c), meshes on the
    leaves. inner = "none": the inner nodes carry no mesh (the pool's chains leave it: split path by default);
    "disabled": they carry a disabled mesh of the same pool (fused path by default, but they are no survivors). Either
    way every 64-survivor tile of leaves needs 64 * (depth - 1) ancestors: far more than its closure can hold."""
    rng = np.random.default_rng(12)
    n = chains * depth
    idx = np.arange(n)
    parent = np.where(idx >= chains, idx - chains, -1).astype(np.int32)
    pos = (rng.uniform(-0.4, 0.4, (n, 3))).astype(np.float32)
    roots = idx < chains
    pos[roots] = np.stack([rng.uniform(-25, 25, chains), rng.uniform(-4, 4, chains), rng.uniform(5, 60, chains)], 1)
    rot = unit_quats(rng, n)
    leaves = idx[idx >= n - chains].astype(np.uint32)
    if inner == "disabled":
        ent = idx.astype(np.uint32)
        enabled = (idx >= n - chains).astype(np.uint8)
        pools = [PoolDesc(RT_OPAQUE, ent, scenes.unit_aabb(n), enabled)]
    else:
        pools = [PoolDesc(RT_OPAQUE, leaves, scenes.unit_aabb(leaves.size))]
    views = view_set(2, "cascades", 0.0)
    return frame_of(scene_from(parent, pos, rot, pools), views, f"interleaved chains ({inner} inner meshes)")


def chain_scene(depths, seed: int = 13, offset: float = 0.03, views=None, name="") -> Frame:
    """One chain per entry of `depths` (a leaf with d ancestors), every node meshed; unit scale, unit quaternions and small
    offsets, so the products stay finite and the walk, not NaN handling, is what is tested."""
    rng = np.random.default_rng(seed)
    parent, roots = [], []
    for d in depths:
        base = len(parent)
        roots.append(base)
        parent += [-1] + list(range(base, base + d))
    n = len(parent)
    pos = rng.uniform(-offset, offset, (n, 3)).astype(np.float32)
    for r, root in enumerate(roots):
        pos[root] = (-12.0 + 8.0 * r, 0.0, 20.0)
    rot = unit_quats(rng, n)
    ent = np.arange(n, dtype=np.uint32)
    pools = [PoolDesc(RT_OPAQUE, ent[ent % 4 != 1], scenes.unit_aabb(int((ent % 4 != 1).sum()))),
             PoolDesc(RT_TRANSLUCENT, ent[ent % 4 == 1], scenes.unit_aabb(int((ent % 4 == 1).sum())))]
    views = view_set(2, "cascades", 0.0) if views is None else views
    return frame_of(scene_from(parent, pos, rot, pools), views, name or f"chains of depth {list(depths)}")


LENGTHS = [1, 4095, 4096, 4097, 12289]


def case_lengths() -> Frame:
    """View 0 sees every slot of the first five pools and only slot 65536 of a 65537-slot pool and slots 1023, 1024, 65535,
    65536 of a 131072-slot pool; view 1 sees nothing. Unseen slots lie behind the camera."""
    rng = np.random.default_rng(14)
    sizes = LENGTHS + [65537, 131072]
    n = sum(sizes)
    seen = np.zeros(n, bool)
    first = np.cumsum([0] + sizes)
    seen[:first[5]] = True
    seen[first[5] + 65536] = True
    seen[first[6] + np.array([1023, 1024, 65535, 65536])] = True
    pos = np.stack([rng.uniform(-3, 3, n), rng.uniform(-3, 3, n), rng.uniform(10, 60, n)], 1).astype(np.float32)
    pos[~seen, 2] *= -1.0
    rot = np.tile(np.array([0, 0, 0, 1], np.float32), (n, 1))
    ent = np.arange(n, dtype=np.uint32)
    pools = [PoolDesc(RT_OPAQUE, ent[first[k]:first[k + 1]], scenes.unit_aabb(sizes[k]), stride=48 + 16 * (k % 2))
             for k in range(len(sizes))]
    views, _ = V.perspective_views([(0.0, 0.0), (np.pi / 2, 0.0)], 1.2, 16 / 9, 0.05)
    return frame_of(scene_from(np.full(n, -1), pos, rot, pools), views, "list lengths at tile boundaries")


def case_equal_keys() -> Frame:
    """Integer lattice, identity rotations, unit scale and an integer camera: every key is an exact integer. 14000 opaque
    entities (plus 2000 nearer) on the eight lattice points at squared distance 50, 2 x 7000 translucent entities on the
    same points (their ties meet in the one descending list: pool order, then slot order), and 5000 UI entities at one z."""
    cam = np.array([3.0, -2.0, 5.0], np.float32)
    shell = np.array([(0, 1, 7), (1, 0, 7), (0, -1, 7), (-1, 0, 7), (3, 4, 5), (4, 3, 5), (-3, 4, 5), (3, -4, 5)], np.float32)
    rng = np.random.default_rng(15)
    groups = [14_000, 2000, 7000, 7000, 5000]
    off = [shell[rng.integers(0, 8, groups[0])], np.tile(np.float32([0, 0, 3]), (groups[1], 1)),
           shell[rng.integers(0, 8, groups[2])], shell[rng.integers(0, 8, groups[3])]]
    pos = [o + cam for o in off]
    ui = np.stack([rng.integers(-30, 30, groups[4]), rng.integers(-5, 5, groups[4]), np.full(groups[4], 4)], 1)
    pos.append(ui.astype(np.float32))
    pos = np.concatenate(pos).astype(np.float32)
    n = pos.shape[0]
    order = rng.permutation(n)  # the groups' entities interleaved in creation order
    pos = pos[order]
    group = np.repeat(np.arange(5), groups)[order]
    rot = np.tile(np.array([0, 0, 0, 1], np.float32), (n, 1))
    ent = np.arange(n, dtype=np.uint32)
    pools = [PoolDesc(RT_OPAQUE, ent[(group == 0) | (group == 1)], scenes.unit_aabb(groups[0] + groups[1])),
             PoolDesc(RT_TRANSLUCENT, ent[group == 2], scenes.unit_aabb(groups[2]), stride=64),
             PoolDesc(RT_TRANSLUCENT, ent[group == 3], scenes.unit_aabb(groups[3])),
             PoolDesc(RT_UI, ent[group == 4], scenes.unit_aabb(groups[4]))]
    views, _ = V.perspective_views([(0.0, 0.0)], 1.3, 16 / 9, 0.05)
    views["uiPlanes"][0] = V.frustum_planes(V.ortho_rev_z((-40.0, 40.0), (-6.0, 6.0), (-50.0, 50.0)))
    views["uiPlaneCount"][0] = 6
    return frame_of(scene_from(np.full(n, -1), pos, rot, pools, cam), views, "equal-key runs")


def case_special_keys() -> Frame:
    """Camera at the origin: entities at the camera (key +0, also from -0), 1e-20 ahead (key 1e-40, subnormal) and 3e19
    ahead (lengthSq3 overflows to +inf), five of each, among ordinary ones, in an ascending and a descending list."""
    rng = np.random.default_rng(16)
    special = np.array([(0, 0, 0), (-0.0, 0, -0.0), (0, 0, 1e-20), (1e-20, 0, 0), (0, 0, 3e19), (1e18, 0, 3e19)], np.float32)
    pos = np.concatenate([np.repeat(special, 5, axis=0),
                          np.stack([rng.uniform(-5, 5, 600), rng.uniform(-3, 3, 600), rng.uniform(2, 40, 600)], 1)])
    pos = pos[rng.permutation(pos.shape[0])].astype(np.float32)
    n = pos.shape[0]
    rot = np.tile(np.array([0, 0, 0, 1], np.float32), (n, 1))
    ent = np.arange(n, dtype=np.uint32)
    pools = [PoolDesc(RT_OPAQUE, ent[ent % 2 == 0], scenes.unit_aabb((n + 1) // 2)),
             PoolDesc(RT_TRANSLUCENT, ent[ent % 2 == 1], scenes.unit_aabb(n // 2))]
    views, _ = V.perspective_views([(0.0, 0.0)], 1.3, 16 / 9, 0.01)
    return frame_of(scene_from(np.full(n, -1), pos, rot, pools), views, "keys +0, subnormal, +inf")


# ---- edge checks (on the oracle's lists or the inputs) -------------------------------------------------------------------
def edge_relocated(f, orun):
    before, larger, unordered, kids = relocation_edges(f)
    assert before > 0 and larger > 0 and unordered > 0, (before, larger, unordered)
    if "reversed" in f.name:
        assert before == kids, "reversed order: every child is stored before its parent"
    assert any((f.t["entity"] == 0)) and all(np.any(m["entity"] == 0) for m in f.pools if m.size)
    assert sum(r.size for _, _, r in lists(orun)) > 0


def edge_views(n):
    def check(f, orun):
        assert f.views.size == n and len(orun.views) == n
        if n > 8:
            high = [v for v in range(8, n) if sum(r.size for w, _, r in lists(orun) if w == v)]
            assert high, "no view >= 8 has a record"
            assert any((m >> 8) and (m & 0xFF) != 0xFF for m in f.masks), "no pool mask with a cleared or set bit >= 8"
    return check


def edge_eight_pools(f, orun):
    assert len(f.pools) == 8 and f.views.size == 16
    if "sparse" in f.name:
        assert any(m.size == 0 for m in f.pools)
        assert orun.views[9]["unsorted"][1][1] == 0 and orun.views[0]["unsorted"][1][1] > 0
        assert orun.views[3]["sorted_counts"][0][0] == 0 and orun.views[12]["sorted_counts"][0][0] > 0
    else:
        # every view holds 6 non-empty unsorted lists and both translucent pools in its descending list
        for v in range(16):
            res = orun.views[v]
            assert len(res["unsorted"]) == 6 and all(c[1] > 0 for c in res["unsorted"]), v
            assert all(c[0] > 0 for c in res["sorted_counts"]), v


def edge_wide_root(f, orun):
    assert int(np.count_nonzero(f.t["parent"] == f.t["entity"][0])) >= 20_000
    assert sum(r.size for _, _, r in lists(orun)) > 20_000


def edge_interleaved(f, orun):
    # distinct ancestors of 64 consecutive leaves (enabled mesh slots) >> the closure of one fused tile
    slot_of = {int(e): i for i, e in enumerate(f.t["entity"])}
    m = f.pools[0]
    leaves = [slot_of[int(e)] for e, on in zip(m["entity"], m["isEnabled"]) if on][:64]
    anc = set()
    for s in leaves:
        p = int(f.t["parent"][s])
        while p:
            anc.add(p)
            p = int(f.t["parent"][slot_of[p]])
    assert len(anc) > 4 * CLOSURE_ENTRIES, len(anc)
    assert orun.views[-1]["unsorted"][0][1] > 64


def chain_depths(t) -> np.ndarray:
    slot_of = np.zeros(int(t["entity"].max()) + 1, np.int64)
    slot_of[t["entity"]] = np.arange(t.size)
    depth = np.zeros(t.size, np.int64)
    p = np.where(t["parent"] != 0, slot_of[t["parent"]], -1)
    while (p >= 0).any():
        depth += p >= 0
        p = np.where(p >= 0, np.where(t["parent"][np.maximum(p, 0)] != 0, slot_of[t["parent"][np.maximum(p, 0)]], -1), -1)
    return depth


def edge_depths(depths):
    def check(f, orun):
        got = set(int(d) for d in chain_depths(f.t))
        assert set(depths) <= got, sorted(set(depths) - got)
        assert sum(r.size for _, _, r in lists(orun)) > sum(depths) // 2
    return check


def edge_lengths(f, orun):
    v0, v1 = orun.views
    assert [c[1] for c in v0["unsorted"]] == LENGTHS + [1, 4]
    assert v0["unsorted"][5][0]["componentOffset"][0] == 65536 * f.pools[5].dtype.itemsize
    assert sorted(v0["unsorted"][6][0]["componentOffset"] // f.pools[6].dtype.itemsize) == [1023, 1024, 65535, 65536]
    assert sum(r.size for _, _, r in lists(types.SimpleNamespace(views=[v1]))) == 0


def edge_equal_keys(f, orun):
    res = orun.views[0]
    assert longest_equal_key_run(res["unsorted"][0][0]) > 3 * SORT_TILE
    trans = res["trans"][0]
    assert longest_equal_key_run(trans) > 3 * SORT_TILE
    assert len(set(trans["bufferIndex"][:3 * SORT_TILE].tolist())) == 2, "the tie run spans both translucent pools"
    assert longest_equal_key_run(res["ui"][0]) > SORT_TILE


def edge_special_keys(f, orun):
    k = all_keys(orun)
    bits = k.view(np.uint32)
    assert np.count_nonzero(bits == 0) >= 10, "keys of exactly +0"
    assert np.count_nonzero((bits > 0) & (bits < 0x00800000)) >= 10, "subnormal keys"
    assert np.count_nonzero(np.isposinf(k)) >= 10, "+inf keys"
    assert not np.isnan(k).any()


DEEP = [254, 255, 256, 300]
CASES = {
    **{f"mixed-relocated-{s}-{o}": (lambda s=s, o=o: case_mixed_relocated(s, o), edge_relocated)
       for s, o in ((21, "random"), (22, "reversed"), (23, "random"), (24, "reversed"))},
    "c3-relocated-random": (lambda: case_c3_relocated("random"), edge_relocated),
    "c3-relocated-reversed": (lambda: case_c3_relocated("reversed"), edge_relocated),
    **{f"views-{n}-{s}": (lambda n=n, s=s: case_views(n, s), edge_views(n))
       for n in (3, 6, 7, 8, 9, 16) for s in ("cascades", "independent")},
    "eight-pools": (lambda: case_eight_pools(False), edge_eight_pools),
    "eight-pools-sparse": (lambda: case_eight_pools(True), edge_eight_pools),
    "wide-root": (case_wide_root, edge_wide_root),
    "interleaved-no-inner-mesh": (lambda: interleaved_chains(inner="none"), edge_interleaved),
    "interleaved-disabled-inner-mesh": (lambda: interleaved_chains(inner="disabled"), edge_interleaved),
    "deep-chains": (lambda: chain_scene(DEEP), edge_depths(DEEP)),
    "deep-chains-relocated": (lambda: relocate(chain_scene(DEEP), 17, "random")[0], edge_depths(DEEP)),
    "list-lengths": (case_lengths, edge_lengths),
    "equal-keys": (case_equal_keys, edge_equal_keys),
    "special-keys": (case_special_keys, edge_special_keys),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_shape_matches_oracle(sceneprep_lib, oracle_built, case):
    build, edge = CASES[case]
    f = build()
    orun = oracle_frame(f)
    edge(f, orun)
    run_gpu(f, orun)


def test_edges_reached_on_the_oracle(oracle_built):
    """The scenes of test_shape_matches_oracle, without a GPU: each still reaches the edge it is named after."""
    for case, (build, edge) in CASES.items():
        f = build()
        edge(f, oracle_frame(f))


def _multiset(f: Frame, orun, inverse):
    """Per list: draw count, and the sorted multiset of (original entity id, key bits, bakedModel bits) of its records."""
    out = {}
    for v, res in enumerate(orun.views):
        for b, (rec, draw, inst) in enumerate(res["unsorted"]):
            out[(v, "u", b)] = (draw, inst)
        out[(v, "sc")] = tuple(res["sorted_counts"])
        for which in ("trans", "ui"):
            out[(v, which)] = res[which][1]
    rows = {}
    for v, name, rec in lists(orun):
        if rec.size == 0:
            continue
        ids = []
        for r in rec:
            m = f.pools[_pool_of(f, v, name, r)]
            ids.append(int(inverse[m["entity"][int(r["componentOffset"]) // m.dtype.itemsize]]))
        keys = rec["distanceSq"].view(np.uint32).astype(np.uint64)
        models = rec["bakedModel"].view(np.uint32)
        rows[(v, name)] = sorted(zip(ids, keys.tolist(), map(bytes, models)))
    return out, rows


def _pool_of(f, v, name, r):
    """Pool of a record: unsorted buffer b belongs to the b-th unsorted pool; a sorted record's bufferIndex counts the
    translucent pools and, in main views, the UI pools (mesh.cpp:341-375)."""
    if name.startswith("unsorted"):
        return [k for k in range(len(f.pools)) if f.rts[k] not in (RT_TRANSLUCENT, RT_UI)][int(name[8:])]
    main = int(f.views[v]["shadowPass"]) < 0
    return [k for k in range(len(f.pools)) if f.rts[k] == RT_TRANSLUCENT or (main and f.rts[k] == RT_UI)][int(r["bufferIndex"])]


@pytest.mark.parametrize("which", ["mixed", "c3"])
def test_relocation_keeps_the_oracle_lists(oracle_built, which):
    """Relocating a scene (relocate: permuted rows, sparse remapped ids, freed slots) changes where records point, never
    what they are: per list the oracle's counts and the multiset of (entity id, key bits, bakedModel bits) are unchanged."""
    if which == "mixed":
        scene = mixed_scene(seed=21, n=1500, max_depth=20, with_ui=True, with_ready=True, box_half=50.0)
        base = frame_of(scene, mixed_views(yaw=2.3), "mixed21")
    else:
        scene = scenes.config_scene("C3", n=8000, seed=77)
        views, _ = V.camera_and_cascades(0.8, -0.1, 1.2, 16 / 9, 0.05, 60.0, (0.1, 0.3, 1.0))
        base = frame_of(scene, views, "C3")
    ident = np.arange(1 << 20, dtype=np.uint32)
    want_counts, want_rows = _multiset(base, oracle_frame(base), ident)
    assert sum(len(r) for r in want_rows.values()) > 100
    for seed, order in ((1, "random"), (2, "reversed")):
        f, id_map = relocate(base, seed, order, freed=25)
        edge_relocated(f, oracle_frame(f))
        inverse = np.zeros(int(id_map.max()) + 1, np.uint32)
        inverse[id_map] = np.arange(id_map.size, dtype=np.uint32)
        got_counts, got_rows = _multiset(f, oracle_frame(f), inverse)
        assert got_counts == want_counts, f"{order}: list counts changed"
        assert got_rows == want_rows, f"{order}: list contents changed"


# ---- a chain deeper than any fixed walk limit: gsp_run, gsp_set_active, gsp_animate -----------------------------------------
@pytest.mark.gpu
def test_chain_of_5000_nodes(sceneprep_lib, oracle_built):
    """One acyclic chain of 5000 transforms (plus a short one), every node meshed. Until the hierarchy was checked for
    cycles once per gsp_set_transforms, every chain walk gave up after 4096 links and gsp_run / gsp_set_active /
    gsp_animate failed with GSP_ERR_HIERARCHY here, although the chain is legal and the oracle walks it."""
    from garden_b200.binding import ScenePrep
    views, _ = V.perspective_views([(0.0, 0.0)], 1.3, 16 / 9, 0.05)
    f = chain_scene([4999, 20], seed=18, offset=0.002, views=views, name="chain of 5000")
    assert int(chain_depths(f.t).max()) == 4999
    t = f.t.copy()
    stride, occ = t.dtype.itemsize, t.size
    raw = t.view(np.uint8).reshape(occ, stride)
    ents = t["entity"].copy()
    o = Oracle()
    sp = ScenePrep(0)
    try:
        stage(sp, f)
        sp.run()
        orun = oracle_frame(f)
        assert orun.views[0]["unsorted"][0][1] > 3000
        compare_frame(sp, f, orun, "chain of 5000")
        # setActive(false) half way down the chain, then on again below: ancestorsActive along 4999 links
        for pick, active in (([2500], False), ([2600, 10], True), ([2500], True)):
            assert o.set_active(raw, stride, occ, ents[pick], active) == 0
            sp.set_active(ents[pick], active)
            got = t.copy()
            sp.writeback_active(got, stride)
            assert np.array_equal(got.view(np.uint8).reshape(occ, stride)[:, 72:74], raw[:, 72:74]), f"setActive {pick}"
            sp.run()
            g = Frame(f"chain of 5000 after setActive {pick} {active}", t, f.pools, f.rts, f.views, f.cam)
            compare_frame(sp, g, oracle_frame(g), g.name)
        # animate position / scale (exact lerp) of nodes near the root: every world matrix below them changes
        pick = np.array([1, 7, 4000])
        flags = np.array([1, 3, 1], np.uint8)
        fa = np.tile(np.float32([0.001, 0.0, 0.001, 1, 1, 1, 0, 0, 0, 1]), (3, 1))
        fb = np.tile(np.float32([-0.001, 0.002, 0.0, 1, 1, 1, 0, 0, 0, 1]), (3, 1))
        tt = np.float32([0.25, 0.5, 0.75])
        assert o.animate(raw, stride, occ, ents[pick], flags, fa, fb, tt) == 0
        sp.animate(ents[pick], flags, fa, fb, tt)
        got = t.copy()
        sp.writeback_trs(got, stride)
        assert np.array_equal(got.view(np.uint8).reshape(occ, stride)[:, 16:48], raw[:, 16:48])
        sp.run()
        g = Frame("chain of 5000 after gsp_animate", t, f.pools, f.rts, f.views, f.cam)
        compare_frame(sp, g, oracle_frame(g), g.name)
    finally:
        sp.close()
        o.close()


@pytest.mark.gpu
def test_cycles_are_refused_and_forgotten(sceneprep_lib):
    """Cycles of every length (a self-parent, 1000 links, a 3000-link chain leading into a 2-cycle) fail gsp_run,
    gsp_set_active and gsp_animate with GSP_ERR_HIERARCHY; the next acyclic gsp_set_transforms clears the state."""
    from garden_b200.binding import GSP_ERR_HIERARCHY, ScenePrep, ScenePrepError
    f = chain_scene([2999, 999, 5], seed=19, offset=0.002)
    ents = f.t["entity"]
    def cyc(pairs):
        t = f.t.copy()
        for child, parent in pairs:
            t["parent"][child] = ents[parent]
        return t
    bad = {"self-parent": cyc([(3005, 3005)]),
           "ring of 1000": cyc([(3000, 3999)]),
           "chain into a 2-cycle": cyc([(0, 1)])}
    sp = ScenePrep(0)
    try:
        for name, t in bad.items():
            g = Frame(name, t, f.pools, f.rts, f.views, f.cam)
            stage(sp, g)
            for call in (sp.run, lambda: sp.set_active(ents[[2]], False),
                         lambda: sp.animate(ents[[2]], np.uint8([1]), np.zeros((1, 10), np.float32),
                                            np.zeros((1, 10), np.float32), np.float32([0.5]))):
                with pytest.raises(ScenePrepError) as e:
                    call()
                assert e.value.code == GSP_ERR_HIERARCHY, name
        stage(sp, f)
        sp.run()
        compare_frame(sp, f, oracle_frame(f), "acyclic again")
    finally:
        sp.close()
