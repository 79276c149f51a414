"""gsp_update_mesh_pool / gsp_update_mesh_pool_indexed: mesh components changed in place (hidden or shown, boxes swapped, ready
counts, destroyed, freed slots reused) must give, frame after frame, exactly what a context gives that staged the same bytes
with gsp_set_mesh_pool: every list with its counts, isVisible, the changed count of the delta write-back, the world matrices
of visible slots and the sorted runs. Each frame is also compared with the oracle on the mutated bytes.

The update links the listed slots without a whole-pool relink: a grown box widens its hierarchy's prepass sphere in place (the
growth cases below fail if it did not: the prepass would drop a slot the oracle lists), a shrunken one keeps the larger sphere.
test_forced_paths re-runs this file with the cull path forced either way and with the prepass off."""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from garden_b200 import scenes, views as V
from garden_b200.scenes import PoolDesc, SceneDesc

from common import OracleRun, compare_gpu_to_oracle
from edge_scenes import mixed_scene, mixed_views

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def raw(m: np.ndarray) -> np.ndarray:
    return m.view(np.uint8).reshape(-1, m.dtype.itemsize)


def clone(m: np.ndarray) -> np.ndarray:
    """Byte copy (ndarray.copy() of a padded struct dtype need not keep the padding bytes)."""
    return np.frombuffer(bytearray(m.tobytes()), dtype=m.dtype)


class World:
    """ECS bytes on the host: the transform pool, the mesh pools, ready counts, component counts, views."""

    def __init__(self, scene: SceneDesc, views, cam=None):
        self.t, pools = scenes.build_aos(scene)
        self.pools = [clone(m) for m in pools]
        self.rts = [p.render_type for p in scene.pools]
        self.ready = [None if p.ready is None else np.ascontiguousarray(p.ready, np.uint8).copy() for p in scene.pools]
        self.counts = [int(m.size) for m in self.pools]
        self.views = views
        self.cam = np.asarray(scene.camera_pos if cam is None else cam, np.float32)

    def stage(self, sp):
        sp.set_transforms(self.t, 80, self.t.size)
        sp.set_pool_count(len(self.pools))
        for k, m in enumerate(self.pools):
            self.set_pool(sp, k)
        sp.set_views(self.views, self.cam)

    def set_pool(self, sp, k):
        m = self.pools[k]
        sp.set_mesh_pool(k, self.rts[k], m, m.dtype.itemsize, m.size, self.counts[k], ready_counts=self.ready[k])

    def oracle(self):
        return OracleRun((self.t, 80, self.t.size), [(m, m.dtype.itemsize, m.size) for m in self.pools], self.rts,
                         self.views, self.cam, ready=self.ready, counts=self.counts)


def c3_world(seed=11):
    scene = scenes.config_scene("C3", n=24_000, seed=seed)   # two pools (opaque + translucent), depth-8 chains: split path
    views, _ = V.perspective_views([(0.7, -0.05)], 1.3, 16 / 9, 0.01)
    return World(scene, views, cam=(2.0, 1.0, -4.0))


def mixed_world(seed=9):
    scene = mixed_scene(seed=seed, n=3000, max_depth=12, with_ui=True, with_ready=True, box_half=50.0)
    return World(scene, mixed_views())


# ---- comparisons ---------------------------------------------------------------------------------------------------------
def copy_to_host(sp, ptr, nbytes) -> np.ndarray:
    out = np.zeros(max(nbytes, 1), np.uint8)
    if nbytes:
        assert sp.lib.gsp_copy_to_host(sp.h, ptr, out.ctypes.data, nbytes) == 0
    return out[:nbytes]


def sorted_runs(sp, w: World):
    """(keys, payloads) of every list of every view, as gsp_get_sorted_run_device hands them out."""
    out = []
    for v in range(w.views.size):
        lists = [(0, b) for b in range(sp.unsorted_buffer_count(v))] + [(1, 0), (2, 0)]
        for kind, b in lists:
            k, p, n = sp.get_sorted_run_device(v, kind, b)
            out.append((copy_to_host(sp, k, 4 * n).tobytes(), copy_to_host(sp, p, 4 * n).view(np.uint32).copy()))
    return out


def lists_of(sp, w: World):
    out = []
    for v in range(w.views.size):
        out += [sp.get_unsorted(v, b) for b in range(sp.unsorted_buffer_count(v))]
        out += [sp.get_sorted_counts(v, b) for b in range(sp.sorted_buffer_count(v))]
        out += [sp.get_sorted(v, 0), sp.get_sorted(v, 1)]
    return out


def assert_same_frame(upd, fresh, w: World, tag: str):
    """Bit for bit: the updated context against a context that staged the same bytes with gsp_set_mesh_pool."""
    a, b = lists_of(upd, w), lists_of(fresh, w)
    assert len(a) == len(b), tag
    for i, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, tuple) and isinstance(x[0], np.ndarray):
            assert x[1:] == y[1:] and x[0].tobytes() == y[0].tobytes(), f"{tag}: list {i} differs"
        else:
            assert x == y, f"{tag}: counts {i} differ"
    ra, rb = sorted_runs(upd, w), sorted_runs(fresh, w)
    assert len(ra) == len(rb)
    seen = [set() for _ in w.pools]
    for (ka, pa), (kb, pb) in zip(ra, rb):
        assert ka == kb and np.array_equal(pa, pb), f"{tag}: sorted runs differ"
        for p in pb:
            seen[int(p) >> 28].add(int(p) & 0x0FFFFFFF)
    for k, m in enumerate(w.pools):
        vis = np.fromiter(seen[k], np.int64) if seen[k] else np.zeros(0, np.int64)
        if vis.size:
            ma, mb = upd.download_models(k, m.size), fresh.download_models(k, m.size)
            assert np.array_equal(ma[vis].view(np.uint32), mb[vis].view(np.uint32)), f"{tag}: pool {k} models differ"


def check_frame(upd, fresh, w: World, tag: str, orun=None):
    """Runs both contexts, compares them with each other and with the oracle, then writes isVisible back through the delta
    path of each into its own copy of the host bytes: same changed counts, same bytes, the oracle's values. The host pools
    then hold those bytes (what both libraries now believe the host holds)."""
    upd.run()
    fresh.run()
    orun = orun or w.oracle()
    compare_gpu_to_oracle(upd, orun, w.rts, w.views, tag)
    assert_same_frame(upd, fresh, w, tag)
    mains = [v for v in range(w.views.size) if int(w.views[v]["shadowPass"]) < 0]
    changed = []
    for k, m in enumerate(w.pools):
        a, b = clone(m), clone(m)
        ca = upd.writeback_visible_delta(k, a, m.dtype.itemsize)
        cb = fresh.writeback_visible_delta(k, b, m.dtype.itemsize)
        assert ca == cb, f"{tag} pool {k}: changed {ca} != {cb}"
        assert a.tobytes() == b.tobytes(), f"{tag} pool {k}: write-back bytes differ"
        if mains:
            want = orun.views[mains[-1]]["visible"][k]
            sel = want != 0xFF
            assert np.array_equal(raw(a)[sel, 15], want[sel]), f"{tag} pool {k}: isVisible differs from the oracle"
        raw(m)[:] = raw(a)
        changed.append(ca)
    return orun, changed


# ---- mutations -----------------------------------------------------------------------------------------------------------
def mutate(w: World, k: int, slots: np.ndarray, rng, live_entities: np.ndarray):
    """Changes the listed slots of pool k in every way an engine does (the host bytes only)."""
    m = w.pools[k]
    r = raw(m)
    for s in slots:
        what = rng.integers(0, 9)
        if what == 0:
            m["isEnabled"][s] ^= 1
        elif what == 1:   # a new box: larger, smaller or moved
            c = rng.normal(0, 1.0, 3).astype(np.float32)
            h = np.abs(rng.normal(0, 1.0, 3)).astype(np.float32) * np.float32(rng.choice([0.1, 1.0, 6.0]))
            m["aabbMin"][s, :3], m["aabbMax"][s, :3] = c - h, c + h
        elif what == 2:   # destroyed: the slot is freed (stale bytes stay)
            m["entity"][s] = 0
        elif what == 3:   # a freed (or live) slot reused by another entity that has a transform
            m["entity"][s] = rng.choice(live_entities)
            m["isEnabled"][s] = 1
        elif what == 4:   # degenerate box
            m["aabbMax"][s, :3] = m["aabbMin"][s, :3]
        elif what == 5:   # NaN box
            m["aabbMin"][s, rng.integers(0, 3)] = np.nan
        elif what == 6 and w.ready[k] is not None:
            w.ready[k][s] = rng.integers(0, 4)
        elif what == 7:   # an entity without a transform, or an id past every transform
            m["entity"][s] = rng.choice([live_entities.max() + 7, rng.integers(1, live_entities.max() + 1)])
        else:
            m["isEnabled"][s] = 1
        if rng.random() < 0.3:
            r[s, 15] = rng.integers(2, 256)  # garbage isVisible byte
    return slots


def push(sp, w: World, k: int, slots=None, first=None, count=None, source="pageable", keep=None):
    """Hands the changed slots to the library: scattered (slots) or as a range, from pageable, pinned or device memory."""
    m = w.pools[k]
    stride = m.dtype.itemsize
    ready = w.ready[k]
    if source == "pageable":  # (the pools themselves are pinned)
        m = clone(m)
        ready = None if ready is None else ready.copy()
    if slots is not None:
        sp.update_mesh_pool_indexed(k, m, stride, slots, w.counts[k], ready)
        return
    if source == "device":
        import torch
        dm = torch.from_numpy(raw(m).copy()).cuda()
        dr = None if w.ready[k] is None else torch.from_numpy(w.ready[k].copy()).cuda()
        keep += [dm, dr]
        sp.update_mesh_pool(k, dm.data_ptr(), stride, first, count, w.counts[k], None if dr is None else dr.data_ptr())
        torch.cuda.synchronize()
    else:
        sp.update_mesh_pool(k, m, stride, first, count, w.counts[k], ready)


def transform_op(step: int, w: World, contexts, rng):
    """The transform-side updates an engine interleaves: indexed TRS updates, gsp_animate, gsp_set_active, a view change. The
    host transform bytes follow through the write-backs, so that the oracle sees the same state."""
    live = np.nonzero(w.t["entity"])[0]
    op = step % 4
    if op == 0:
        sel = rng.choice(live, size=max(1, live.size // 40), replace=False).astype(np.uint32)
        w.t["position"][sel] += rng.normal(0, 0.5, (sel.size, 3)).astype(np.float32)
        for sp in contexts:
            sp.update_transforms_indexed(w.t, 80, sel)
    elif op == 1:
        sel = rng.choice(live, size=max(1, live.size // 50), replace=False)
        ids = w.t["entity"][sel].astype(np.uint32)
        fa = np.concatenate([w.t["position"][sel], w.t["scale"][sel], w.t["rotation"][sel]], axis=1).astype(np.float32)
        fb = fa.copy()
        fb[:, :3] += np.float32(1.5)
        tt = rng.random(ids.size).astype(np.float32)
        flags = np.full(ids.size, 7, np.uint8)
        for sp in contexts:
            sp.animate(ids, flags, fa, fb, tt)
        contexts[-1].writeback_trs(w.t, 80)
    elif op == 2:
        ids = w.t["entity"][rng.choice(live, size=max(1, live.size // 100), replace=False)].astype(np.uint32)
        active = bool(step % 8 == 2)
        for sp in contexts:
            sp.set_active(ids, active)
        contexts[-1].writeback_active(w.t, 80)
    else:
        views = w.views.copy()
        turn = V.perspective_views([(0.7 + 0.1 * step, -0.05)], 1.3, 16 / 9, 0.01)[0][0]
        main = int(np.nonzero(views["shadowPass"] < 0)[0][-1])
        views[main]["planes"] = turn["planes"]
        w.views = views
        for sp in contexts:
            sp.set_views(w.views, w.cam)


# ---- multi-frame sequences -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["c3", "mixed"])
def test_mutation_sequences_match_a_fresh_staging(sceneprep_lib, oracle_built, which):
    import torch  # noqa: F401  (device sources)
    from garden_b200.binding import ScenePrep, pin_host, unpin_host
    w = c3_world() if which == "c3" else mixed_world()
    rng = np.random.default_rng(1 if which == "c3" else 2)
    live = w.t["entity"][w.t["entity"] != 0].astype(np.uint32)
    upd, fresh = ScenePrep(0), ScenePrep(0)
    pinned = [m for m in w.pools if m.size] + [r for r in w.ready if r is not None and r.size]
    for a in pinned:
        pin_host(a)
    keep = []
    try:
        w.stage(upd)
        w.stage(fresh)
        check_frame(upd, fresh, w, f"{which} frame 0")
        sources = ["pageable", "pinned", "device"]
        total_changed = []
        for frame in range(1, 13):
            if frame % 3 == 1:
                transform_op(frame, w, [upd, fresh], rng)       # a full chain pass is pending: the update skips its walk
            for k, m in enumerate(w.pools):
                if m.size == 0:
                    continue
                n = max(1, m.size * 3 // 100)
                if frame % 2:  # scattered, shuffled, with duplicates
                    slots = rng.choice(m.size, size=n, replace=False).astype(np.uint32)
                    mutate(w, k, slots, rng, live)
                    dup = rng.choice(slots, size=max(1, n // 5))
                    slots = rng.permutation(np.concatenate([slots, dup])).astype(np.uint32)
                    push(upd, w, k, slots=slots, source=sources[(frame // 2) % 2])
                else:          # a dirty range, from each kind of memory in turn
                    first = int(rng.integers(0, max(1, m.size - 4 * n)))
                    count = min(m.size - first, 4 * n)
                    mutate(w, k, first + rng.choice(count, size=min(n, count), replace=False), rng, live)
                    push(upd, w, k, first=first, count=count, source=sources[(frame // 2) % 3], keep=keep)
                w.set_pool(fresh, k)
            if frame % 3 == 2:
                transform_op(frame, w, [upd, fresh], rng)       # after the update: the incremental chain bounds stand
            _, changed = check_frame(upd, fresh, w, f"{which} frame {frame}")
            total_changed.append(sum(changed))
        assert sum(total_changed) > 0
    finally:
        upd.close(); fresh.close()
        for a in pinned:
            unpin_host(a)


# ---- growth: the prepass sphere must follow a grown box ------------------------------------------------------------------
FAR = 3000.0
P_POS = (0.0, 6 * FAR, 0.0)  # the parent of the modelWithAncestors == false transform


def growth_world():
    """A small C3-shaped scene plus hierarchies with tiny boxes high above the camera, outside the view (the perspective view
    reaches to infinity, so they are not placed along it): a lone root (entity A), a chain of 12 links (leaf L), a transform
    with modelWithAncestors == false (entity F) under a parent P placed much higher still, and a lone root in a fourth place
    (entity R). F's prepass record takes F's own position and bound, not its hierarchy's sphere about P, and only that record
    can reach the view (test_growth_reaches_the_view checks the distances). Pool 0 gets one slot on A, L and F, and one on
    the chain's root that is later re-pointed to R."""
    base = scenes.config_scene("C3", n=6000, seed=5)
    n0 = base.entity_count
    pos = [(30, FAR, 0)] + [(-30, FAR, 0)] + [(0.5, 0, 0)] * 12 + [(0, FAR, 30), (0, FAR, -30), P_POS]
    parent = [-1, -1] + [n0 + 1 + i for i in range(12)] + [n0 + 16, -1, -1]
    tfl = [3, 3] + [3] * 12 + [1, 3, 3]
    extra = len(pos)
    position = np.concatenate([base.position, np.asarray(pos, np.float32)])
    rotation = np.concatenate([base.rotation, np.tile(np.array([0, 0, 0, 1], np.float32), (extra, 1))])
    scale = np.concatenate([base.scale, np.ones((extra, 3), np.float32)])
    par = np.concatenate([base.parent, np.asarray(parent, np.int32)])
    tflags = np.concatenate([base.tflags, np.asarray(tfl, np.uint8)])
    ent = {"A": n0, "L": n0 + 13, "F": n0 + 14, "R": n0 + 15, "chain_root": n0 + 1, "P": n0 + 16}
    p0 = base.pools[0]
    tiny = np.array([[-0.05, -0.05, -0.05, 0.05, 0.05, 0.05]] * 4, np.float32)
    owners = np.array([ent["A"], ent["L"], ent["F"], ent["chain_root"]], np.uint32)
    pools = [PoolDesc(p0.render_type, np.concatenate([p0.entity_index, owners]), np.concatenate([p0.aabb, tiny]))] + base.pools[1:]
    scene = SceneDesc(position, rotation, scale, par, tflags, pools, None, np.array([2.0, 1.0, -4.0], np.float32), "growth")
    views, _ = V.perspective_views([(0.7, -0.05)], 1.3, 16 / 9, 0.01)
    w = World(scene, views)
    first = p0.entity_index.size
    return w, {"A": first, "L": first + 1, "F": first + 2, "repoint": first + 3}, ent


def listed(orun, pool_stride, slot) -> bool:
    """The slot is in some list of the oracle's frame (pool 0 is the only opaque pool)."""
    off = slot * pool_stride
    for res in orun.views:
        for rec, _, _ in res["unsorted"]:
            if (rec["componentOffset"] == off).any():
                return True
    return False


def box_at(world_centre, owner_pos, half=12.0):
    c = np.asarray(world_centre, np.float32) - np.asarray(owner_pos, np.float32)
    return c - np.float32(half), c + np.float32(half)


def test_growth_reaches_the_view(sceneprep_lib, oracle_built):
    from garden_b200.binding import ScenePrep
    w, slot, ent = growth_world()
    m = w.pools[0]
    stride = m.dtype.itemsize
    target = (0.0, 0.0, 0.0)  # around the camera: inside the view
    upd, fresh = ScenePrep(0), ScenePrep(0)
    try:
        w.stage(upd)
        w.stage(fresh)
        orun, _ = check_frame(upd, fresh, w, "growth start")
        for s in slot.values():
            assert not listed(orun, stride, s), "the far slots start outside the view"
        leaf_pos = (-30 + 6.0, FAR, 0)
        # F's hierarchy sphere is centred on P, with a radius of about |F's position| + the grown box's reach (both ~FAR):
        # it cannot hold the view, so F is listed only if its own-bound record (kChainRecords, !modelWithAncestors) grew
        f_pos = np.array([0, FAR, 30], np.float64)
        reach = np.linalg.norm(f_pos) + np.linalg.norm(np.array(target) - f_pos) + 12 * np.sqrt(3)
        assert w.t["parent"][ent["F"]] == ent["P"] + 1 and w.t["modelWithAncestors"][ent["F"]] == 0
        assert np.linalg.norm(np.array(P_POS) - np.array(target)) > 1.4 * reach
        cases = [("lone root", slot["A"], None, (30, FAR, 0)),
                 ("deep leaf", slot["L"], None, leaf_pos),
                 ("model without ancestors", slot["F"], None, (0, FAR, 30)),
                 ("re-pointed to another hierarchy", slot["repoint"], ent["R"], (0, FAR, -30))]
        for i, (name, s, new_entity, owner) in enumerate(cases):
            lo, hi = box_at(target, owner)
            m["aabbMin"][s, :3], m["aabbMax"][s, :3] = lo, hi
            if new_entity is not None:
                m["entity"][s] = new_entity + 1
            if i % 2:
                upd.update_mesh_pool(0, m, stride, s, 1, w.counts[0])
            else:
                upd.update_mesh_pool_indexed(0, m, stride, [s], w.counts[0])
            w.set_pool(fresh, 0)
            orun, _ = check_frame(upd, fresh, w, f"growth: {name}")
            assert listed(orun, stride, s), f"{name}: the grown box must reach the view"
        # shrinking: the lone root's box goes back to a speck far away; the kept larger sphere must not change the lists
        s = slot["A"]
        m["aabbMin"][s, :3], m["aabbMax"][s, :3] = -0.05, 0.05
        upd.update_mesh_pool_indexed(0, m, stride, [s], w.counts[0])
        w.set_pool(fresh, 0)
        orun, _ = check_frame(upd, fresh, w, "shrink")
        assert not listed(orun, stride, s), "the shrunken box is out of the view again"
    finally:
        upd.close(); fresh.close()


# ---- a range whose components and ready counts both go through the scratch buffer -----------------------------------------
def test_pageable_range_with_ready_counts_grows_the_scratch(sceneprep_lib, oracle_built):
    """Components and ready counts of a range both in pageable memory share the device scratch buffer. Everything here is
    first staged from pinned memory, so the scratch buffer is empty when the first update arrives; the second update is far
    larger than the first. Both must see the bytes of this call (a scratch buffer reallocated between the two copies would
    leave the components' pointer in freed memory)."""
    from garden_b200.binding import ScenePrep, pin_host, unpin_host
    scene = scenes.config_scene("C2", n=200_000, seed=8)
    scene.pools[0].ready = np.ones(scene.pools[0].entity_index.size, np.uint8)
    views, _ = V.camera_and_cascades(0.3, -0.1, 1.2, 16 / 9, 0.01, 100.0, (0.05, 0.1, 0.25, 1.0))
    w = World(scene, views, cam=(1.0, 0.5, -2.0))
    m, ready = w.pools[0], w.ready[0]
    stride = m.dtype.itemsize
    pinned = [w.t, m, ready]
    for a in pinned:
        pin_host(a)
    rng = np.random.default_rng(12)
    upd, fresh = ScenePrep(0), ScenePrep(0)
    try:
        w.stage(upd)
        w.stage(fresh)
        check_frame(upd, fresh, w, "pinned staging")
        for first, count in ((100, 16), (0, m.size)):
            sel = first + rng.choice(count, size=max(1, count // 3), replace=False)
            ready[sel] = 0                                        # not ready: leaves every list
            m["aabbMax"][sel[::2], :3] *= np.float32(3.0)         # grown boxes
            upd.update_mesh_pool(0, clone(m), stride, first, count, w.counts[0], ready.copy())  # both pageable
            w.set_pool(fresh, 0)
            check_frame(upd, fresh, w, f"pageable range [{first}, {first + count})")
    finally:
        upd.close(); fresh.close()
        for a in pinned:
            unpin_host(a)


# ---- launches ------------------------------------------------------------------------------------------------------------
def test_next_frame_launches_what_an_unchanged_frame_launches(sceneprep_lib, oracle_built):
    from garden_b200.binding import ScenePrep
    w, slot, _ = growth_world()
    m = w.pools[0]
    stride = m.dtype.itemsize
    sp = ScenePrep(0)
    try:
        w.stage(sp)
        sp.run()
        sp.run()
        steady = sp.last_launch_count()
        rng = np.random.default_rng(4)
        flip = rng.choice(m.size - 8, size=m.size // 100, replace=False).astype(np.uint32)
        m["isEnabled"][flip] ^= 1
        sp.update_mesh_pool_indexed(0, m, stride, flip, w.counts[0])
        sp.run()
        assert sp.last_launch_count() == steady, "flag update"
        lo, hi = box_at((0, 0, 0), (30, FAR, 0))
        m["aabbMin"][slot["A"], :3], m["aabbMax"][slot["A"], :3] = lo, hi
        sp.update_mesh_pool(0, m, stride, slot["A"], 1, w.counts[0])
        sp.run()
        assert sp.last_launch_count() == steady, "growing update"
        compare_gpu_to_oracle(sp, w.oracle(), w.rts, w.views, "launches")
        w.set_pool(sp, 0)
        sp.run()
        assert sp.last_launch_count() > steady, "gsp_set_mesh_pool relinks"
    finally:
        sp.close()


# ---- state ---------------------------------------------------------------------------------------------------------------
def test_snapshot_and_component_count(sceneprep_lib, oracle_built):
    from garden_b200.binding import GSP_ERR_STATE, ScenePrep, ScenePrepError
    w = c3_world(seed=3)
    m = w.pools[1]
    stride = m.dtype.itemsize
    sp, fresh = ScenePrep(0), ScenePrep(0)
    try:
        w.stage(sp)
        w.stage(fresh)
        check_frame(sp, fresh, w, "state start")
        sp.run()
        before = [sp.get_unsorted(0, 0)[0].copy(), sp.get_sorted(0, 0)[0].copy()]
        sp.fetch_all_async()
        raw(m)[: m.size // 2, 15] = 0
        m["isEnabled"][: m.size // 2] = 0
        sp.update_mesh_pool(1, m, stride, 0, m.size // 2, w.counts[1])
        during = [sp.get_unsorted(0, 0)[0], sp.get_sorted(0, 0)[0]]
        for a, b in zip(before, during):
            assert a.tobytes() == b.tobytes(), "the snapshot survives an update"
        with pytest.raises(ScenePrepError) as e:
            sp.sync()  # the update ended the frame's results
        assert e.value.code == GSP_ERR_STATE
        w.set_pool(fresh, 1)
        check_frame(sp, fresh, w, "after the snapshot")
        # componentCount 0: the pool leaves every list (new layout: the snapshot ends), isVisible stays the host's
        sp.run()
        sp.fetch_all_async()
        w.counts[1] = 0
        sp.update_mesh_pool_indexed(1, m, stride, [0], 0)
        with pytest.raises(ScenePrepError) as e:
            sp.get_unsorted(0, 0)
        assert e.value.code == GSP_ERR_STATE
        raw(m)[:, 15] = 9
        w.set_pool(fresh, 1)
        orun, changed = check_frame(sp, fresh, w, "count 0")
        assert changed[1] == 0 and (raw(m)[:, 15] == 9).all()
        assert all((orun.views[v]["visible"][1] == 0xFF).all() for v in range(w.views.size) if "visible" in orun.views[v])
        w.counts[1] = m.size
        sp.update_mesh_pool(1, m, stride, 0, m.size, w.counts[1])  # (the host's isVisible bytes are all 9 now)
        w.set_pool(fresh, 1)
        check_frame(sp, fresh, w, "count back")
    finally:
        sp.close(); fresh.close()


def test_refusals_change_nothing(sceneprep_lib, oracle_built):
    import torch
    from garden_b200.binding import GSP_ERR_INVALID, GSP_ERR_STATE, ScenePrep, ScenePrepError
    w = mixed_world(seed=4)
    k_ready = next(k for k, r in enumerate(w.ready) if r is not None)
    k_plain = next(k for k, r in enumerate(w.ready) if r is None and w.pools[k].size)
    sp = ScenePrep(0)
    try:
        w.stage(sp)
        sp.run()
        want = lists_of(sp, w)
        mr, mp = w.pools[k_ready], w.pools[k_plain]
        sr, spl = mr.dtype.itemsize, mp.dtype.itemsize
        # the bytes change, so an update that went through would change the next frame
        for m in (mr, mp):
            m["isEnabled"][:] = 0
        dev = torch.from_numpy(raw(mp).copy()).cuda()
        lib, h = sp.lib, sp.h
        slots = np.arange(4, dtype=np.uint32)
        calls = [
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, 8, mp.ctypes.data, spl, 0, 1, mp.size, None)),
            (GSP_ERR_STATE, lambda: lib.gsp_update_mesh_pool(h, len(w.pools), mp.ctypes.data, spl, 0, 1, 1, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, k_plain, mp.ctypes.data, spl + 16, 0, 1, mp.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, k_plain, mp.ctypes.data, spl, mp.size - 1, 2, mp.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool_indexed(h, k_plain, mp.ctypes.data, spl,
                                                                       np.array([0, mp.size], np.uint32).ctypes.data, 2, mp.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, k_plain, mp.ctypes.data, spl, 0, 1, mp.size,
                                                               w.ready[k_ready].ctypes.data)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, k_ready, mr.ctypes.data, sr, 0, 1, mr.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool(h, k_plain, None, spl, 0, 1, mp.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool_indexed(h, k_plain, mp.ctypes.data, spl, None, 1, mp.size, None)),
            (GSP_ERR_INVALID, lambda: lib.gsp_update_mesh_pool_indexed(h, k_plain, dev.data_ptr(), spl, slots.ctypes.data, 4,
                                                                       mp.size, None)),
        ]
        for i, (code, call) in enumerate(calls):
            assert call() == code, f"refusal {i}: {lib.gsp_last_error(h).decode()}"
            sp.run()
            got = lists_of(sp, w)
            for x, y in zip(got, want):
                if isinstance(x, tuple) and isinstance(x[0], np.ndarray):
                    assert x[1:] == y[1:] and x[0].tobytes() == y[0].tobytes(), f"refusal {i} changed the next frame"
                else:
                    assert x == y, f"refusal {i} changed the next frame"
        # count == 0 is a no-op, even with null pointers
        assert lib.gsp_update_mesh_pool(h, k_plain, None, spl, 0, 0, mp.size, None) == 0
        assert lib.gsp_update_mesh_pool_indexed(h, k_plain, None, spl, None, 0, mp.size, None) == 0
        with pytest.raises(ScenePrepError):
            sp.update_mesh_pool(k_plain, mp, spl + 16, 0, 1, mp.size)
    finally:
        sp.close()


# ---- forced paths --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env", [{"GSP_SPLIT": "0"}, {"GSP_SPLIT": "1"}, {"GSP_PREPASS": "0"}], ids=["fused", "split", "no-prepass"])
def test_forced_paths(sceneprep_lib, oracle_built, env):
    if os.environ.get("GSP_MESH_UPDATE_CHILD"):
        pytest.skip("already forced")
    res = subprocess.run([sys.executable, "-m", "pytest", __file__, "-m", "gpu", "-x", "-q", "-k", "not forced_paths"],
                         cwd=ROOT, env={**os.environ, **env, "GSP_MESH_UPDATE_CHILD": "1"}, capture_output=True, text=True,
                         timeout=1500)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-1000:]
