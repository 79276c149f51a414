"""GPU test of the gather + k-way merge, with the ranks emulated on one device: R shards of one scene are prepared one
after the other, their runs concatenated the way the NCCL all-gather would lay them out, and every rank's merged
key-range slice is checked against (a) the numpy statement of the merge and (b) a single-GPU sort of the whole scene."""
import numpy as np
import pytest

from garden_b200 import scenes, views as V
from garden_b200.dist import merge_reference, plan_from_blocks, plan_gather

pytestmark = pytest.mark.gpu


def _prepare(sp, scene, views):
    t, pools = scenes.build_aos(scene)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, scene.pools[k].render_type, m, m.dtype.itemsize, m.size)
    sp.set_views(views, scene.camera_pos)
    sp.run()


def _runs_to_host(sp, torch):
    counts = sp.list_counts().astype(np.int64)
    total = int(counts.sum())
    k = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    p = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    sp.export_runs(k.data_ptr(), p.data_ptr(), max(total, 1))
    sp.sync()
    torch.cuda.synchronize()
    return counts, k[:total].cpu().numpy().view(np.uint32), p[:total].cpu().numpy().view(np.uint32)


def _shards(whole, ranks, chains, depth):
    n = whole.entity_count
    per = (chains // ranks) * (depth + 1)
    starts = [r * per for r in range(ranks)] + [n]
    out = []
    for r in range(ranks):
        a, b = starts[r], starts[r + 1]
        out.append(scenes.SceneDesc(whole.position[a:b], whole.rotation[a:b], whole.scale[a:b],
                                    np.where(whole.parent[a:b] >= 0, whole.parent[a:b] - a, -1).astype(np.int32), whole.tflags[a:b],
                                    [scenes.PoolDesc(whole.pools[0].render_type, np.arange(b - a, dtype=np.uint32), whole.pools[0].aabb[a:b])],
                                    None, whole.camera_pos))
    return out, starts


@pytest.mark.parametrize("ranks", [1, 2, 3, 4, 5, 6, 7, 8, 16])
def test_packed_exchange_emulated_ranks(sceneprep_lib, ranks):
    """The host-synchronisation-free exchange (gsp_export_runs_packed -> [all-gather] -> gsp_merge_gathered_packed_tree):
    blocks are exported right after gsp_run_async (no gsp_sync), laid out as the all-gather would, merged per rank, and
    checked against the numpy merge and against a single sort of the whole scene. Then the overflow protocol."""
    import torch
    from garden_b200.binding import ScenePrep
    chains, depth = 3000, 4
    n = chains * (depth + 1)
    whole = scenes.make_scene(n, depth, 11, (-150, -10, -150, 150, 10, 150))
    whole.camera_pos = np.array([2.0, 1.0, -3.0], np.float32)
    views, _ = V.camera_and_cascades(0.3, -0.1, 1.2, 16 / 9, 0.01, 100.0, (0.05, 0.1, 0.25, 1.0))
    sp = ScenePrep(0)
    _prepare(sp, whole, views)
    full_counts, full_k, full_p = _runs_to_host(sp, torch)
    lists = full_counts.size
    lib = sp.lib
    cap = int(full_counts.sum())  # plenty for every shard
    words = lib.gsp_exchange_block_words(cap)
    gathered = torch.zeros(words * ranks, dtype=torch.int32, device="cuda")
    shards, starts = _shards(whole, ranks, chains, depth)
    shard_runs = []
    for r, sc in enumerate(shards):
        t, pools = scenes.build_aos(sc)
        sp.set_transforms(t, t.dtype.itemsize, t.size)
        sp.set_pool_count(len(pools))
        for k, m in enumerate(pools):
            sp.set_mesh_pool(k, sc.pools[k].render_type, m, m.dtype.itemsize, m.size)
        sp.set_views(views, sc.camera_pos)
        sp.run_async()  # no sync: the export reads the list lengths on the device
        sp.export_runs_packed(gathered[r * words:].data_ptr(), cap)
        sp.sync()
        shard_runs.append(_runs_to_host(sp, torch))
    torch.cuda.synchronize()
    hdr = gathered.cpu().numpy().view(np.uint32).reshape(ranks, words)[:, :8 + lists]
    all_counts = np.stack([c for c, _, _ in shard_runs])
    assert np.array_equal(hdr[:, 8:8 + lists].astype(np.int64), all_counts)
    assert np.all(hdr[:, 0] == 0x47535031) and np.all(hdr[:, 1] == lists) and np.all(hdr[:, 4] == 0)
    offsets, _, out_offsets, totals = plan_gather(all_counts)
    total = int(totals.sum())
    plan = torch.zeros(lib.gsp_merge_plan_words(ranks, lists), dtype=torch.int32, device="cuda")
    merged_k = np.zeros(total, np.uint32); merged_p = np.zeros(total, np.uint32); merged_r = np.zeros(total, np.uint8)
    covered = np.zeros(total, bool)
    for me in range(ranks):
        out_k = torch.zeros(total, dtype=torch.int32, device="cuda"); out_p = torch.zeros_like(out_k)
        out_r = torch.zeros(total, dtype=torch.uint8, device="cuda")
        sinfo = torch.zeros(lists * 2, dtype=torch.int32, device="cuda")
        # (scratch poisoned so stale reads would show)
        scratch = torch.full((int(lib.gsp_merge_tree_scratch_words(total)),), -1, dtype=torch.int32, device="cuda")
        rc = lib.gsp_merge_gathered_packed_tree(0, ranks, me, lists, cap, gathered.data_ptr(), plan.data_ptr(), sinfo.data_ptr(),
                                                out_k.data_ptr(), out_p.data_ptr(), out_r.data_ptr(), total, scratch.data_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        pl = plan.cpu().numpy().view(np.uint32)
        assert pl[-8] == 0 and pl[-7] == total and pl[-6] == all_counts.sum(axis=1).max()
        assert np.array_equal(pl[2 * ranks * lists: 2 * ranks * lists + lists], out_offsets)
        # the device plan equals the numpy statement of kMergePlan (which the gloo CPU test exercises)
        e_off, e_cnt, e_out, e_flags = plan_from_blocks(gathered.cpu().numpy().view(np.uint32), ranks, lists, cap, total)
        assert np.array_equal(pl[:ranks * lists].reshape(ranks, lists), e_off) and np.array_equal(pl[ranks * lists:2 * ranks * lists].reshape(ranks, lists), e_cnt)
        assert np.array_equal(pl[2 * ranks * lists: 2 * ranks * lists + lists], e_out) and np.array_equal(pl[-8:].astype(np.int64), e_flags)
        info = sinfo.cpu().numpy().reshape(lists, 2)
        ok, op, orr = out_k.cpu().numpy().view(np.uint32), out_p.cpu().numpy().view(np.uint32), out_r.cpu().numpy()
        for l in range(lists):
            start, length = int(info[l, 0]), int(info[l, 1])
            runs_k = [shard_runs[r][1][offsets[r, l]: offsets[r, l] + all_counts[r, l]] for r in range(ranks)]
            runs_p = [shard_runs[r][2][offsets[r, l]: offsets[r, l] + all_counts[r, l]] for r in range(ranks)]
            ek, ep, er, estart = merge_reference(runs_k, runs_p, my_rank=me)
            assert (start, length) == (estart, ek.size), f"rank {me} list {l}: slice bounds"
            o = int(out_offsets[l])
            assert np.array_equal(ok[o:o + length], ek) and np.array_equal(op[o:o + length], ep) and np.array_equal(orr[o:o + length], er)
            g = slice(o + start, o + start + length)
            assert not covered[g].any()
            covered[g] = True
            merged_k[g], merged_p[g], merged_r[g] = ek, ep, er
    assert covered.all()
    global_p = (merged_p & 0xF0000000) | ((merged_p & 0x0FFFFFFF) + np.array(starts, np.uint32)[merged_r])
    assert np.array_equal(merged_k, full_k) and np.array_equal(global_p, full_p)

    # overflow protocol: a block that cannot hold the rank's lists is flagged, carries nothing, and the merge reports it
    small = max(int(all_counts.sum(axis=1).max()) // 2, 1)
    words_s = lib.gsp_exchange_block_words(small)
    g2 = torch.zeros(words_s * ranks, dtype=torch.int32, device="cuda")
    sp.run_async()
    for r in range(ranks):
        sp.export_runs_packed(g2[r * words_s:].data_ptr(), small)  # (the last shard, into every block)
    sentinel = torch.full((total,), 0x5a5a5a5a, dtype=torch.int32, device="cuda")
    out_p = sentinel.clone(); out_r = torch.zeros(total, dtype=torch.uint8, device="cuda")
    sinfo = torch.zeros(lists * 2, dtype=torch.int32, device="cuda")
    scratch = torch.zeros(int(lib.gsp_merge_tree_scratch_words(total)), dtype=torch.int32, device="cuda")
    rc = lib.gsp_merge_gathered_packed_tree(0, ranks, 0, lists, small, g2.data_ptr(), plan.data_ptr(), sinfo.data_ptr(),
                                            sentinel.data_ptr(), out_p.data_ptr(), out_r.data_ptr(), total, scratch.data_ptr())
    assert rc == 0
    sp.sync()
    torch.cuda.synchronize()
    pl = plan.cpu().numpy().view(np.uint32)
    assert pl[-8] & 1, "overflow must be reported"
    assert pl[-6] == int(shard_runs[-1][0].sum()), "the needed capacity is reported"
    assert bool((sentinel == 0x5a5a5a5a).all()), "nothing may be merged from an overflowed exchange"
    assert int(sinfo.cpu().numpy().reshape(lists, 2)[:, 1].sum()) == 0
    sp.close()


@pytest.mark.parametrize("ranks,key_bits,lists", [(2, 32, 3), (3, 6, 3), (4, 20, 3), (7, 3, 3), (8, 32, 3), (16, 10, 3), (8, 12, 40), (5, 4, 97),
                                                   (32, 10, 128)])
def test_merge_tree_synthetic_runs(sceneprep_lib, ranks, key_bits, lists):
    """The merge-path tree on hand-made blocks: runs of very different lengths (some empty, some spanning many 2048-element
    tiles), few distinct keys (ties decide by rank, then by position in the run) or 32-bit keys. Every rank's slice has to
    equal the numpy merge, and the slices together have to tile every list."""
    import torch
    from garden_b200.binding import load_library
    lib = load_library()
    rng = np.random.default_rng(1000 * ranks + key_bits + lists)
    # (many lists: the (list, pair) job table spans several warp-scan rounds; some lists are empty on every rank. 128 lists
    # at 32 ranks, the largest layout at the largest rank count, fill all 2048 jobs of level 1 with short runs)
    lengths = rng.integers(0, 60000 if lists <= 3 else 5000 if lists <= 100 else 600, size=(ranks, lists))
    lengths[rng.integers(0, ranks), 0] = 0            # an empty run
    lengths[:, 2] = rng.integers(0, 40, size=ranks)   # a list shorter than one tile
    if ranks >= 3:
        lengths[1, 1] = 150000                        # one rank dominates a list
    if lists > 3:
        lengths[:, 5::7] = 0                          # lists nobody has anything in
    cap = int(lengths.sum(axis=1).max()) + 17
    words = lib.gsp_exchange_block_words(cap)
    blocks = np.zeros((ranks, words), np.uint32)
    runs = [[None] * lists for _ in range(ranks)]
    for r in range(ranks):
        blocks[r, :5] = (0x47535031, lists, int(lengths[r].sum()), cap, 0)
        at = 0
        for l in range(lists):
            n = int(lengths[r, l])
            k = np.sort(rng.integers(0, 1 << key_bits, size=n, dtype=np.uint64).astype(np.uint32))
            p = rng.integers(0, 1 << 28, size=n, dtype=np.uint64).astype(np.uint32)
            p = p[np.lexsort((p, k))]  # runs are tie-ordered by payload, as the stable device sort leaves them
            blocks[r, 8 + l] = n
            blocks[r, 256 + at:256 + at + n] = k
            blocks[r, 256 + cap + at:256 + cap + at + n] = p
            runs[r][l] = (k, p)
            at += n
    total = int(lengths.sum())
    gathered = torch.from_numpy(blocks.view(np.int32).reshape(-1)).cuda()
    plan = torch.zeros(lib.gsp_merge_plan_words(ranks, lists), dtype=torch.int32, device="cuda")
    out_offsets = np.concatenate([[0], np.cumsum(lengths.sum(axis=0))[:-1]])
    covered = np.zeros(total, bool)
    for me in range(ranks):
        out_k = torch.full((total,), -1, dtype=torch.int32, device="cuda"); out_p = out_k.clone()
        out_r = torch.full((total,), 255, dtype=torch.uint8, device="cuda")
        sinfo = torch.zeros(lists * 2, dtype=torch.int32, device="cuda")
        scratch = torch.full((int(lib.gsp_merge_tree_scratch_words(total)),), -1, dtype=torch.int32, device="cuda")
        rc = lib.gsp_merge_gathered_packed_tree(0, ranks, me, lists, cap, gathered.data_ptr(), plan.data_ptr(), sinfo.data_ptr(),
                                                out_k.data_ptr(), out_p.data_ptr(), out_r.data_ptr(), total, scratch.data_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        assert plan.cpu().numpy().view(np.uint32)[-8] == 0
        info = sinfo.cpu().numpy().reshape(lists, 2)
        ok, op, orr = out_k.cpu().numpy().view(np.uint32), out_p.cpu().numpy().view(np.uint32), out_r.cpu().numpy()
        for l in range(lists):
            ek, ep, er, estart = merge_reference([runs[r][l][0] for r in range(ranks)], [runs[r][l][1] for r in range(ranks)], my_rank=me)
            start, length = int(info[l, 0]), int(info[l, 1])
            assert (start, length) == (estart, ek.size), f"rank {me} list {l}: slice bounds"
            o = int(out_offsets[l])
            assert np.array_equal(ok[o:o + length], ek), f"rank {me} list {l}: keys"
            assert np.array_equal(op[o:o + length], ep), f"rank {me} list {l}: payloads"
            assert np.array_equal(orr[o:o + length], er), f"rank {me} list {l}: ranks"
            assert not covered[o + start:o + start + length].any()
            covered[o + start:o + start + length] = True
    assert covered.all()


def test_merge_tree_refuses_what_it_cannot_index(sceneprep_lib):
    """gsp_merge_gathered_packed_tree refuses (GSP_ERR_INVALID, before anything is launched) gathered blocks that reach 2^32
    words, which its 32-bit element indices cannot address, and more (list, pair of runs) jobs than its table holds. The
    buffers are tiny placeholders: a refused call reads none of them."""
    import torch
    from garden_b200.binding import GSP_ERR_INVALID, load_library
    lib = load_library()
    d = torch.zeros(64, dtype=torch.int32, device="cuda").data_ptr()
    cap = (1 << 30) - 128  # (256 + 2 * cap) * 2 ranks = 2^32 words
    assert (256 + 2 * cap) * 2 == 1 << 32
    assert lib.gsp_merge_gathered_packed_tree(0, 2, 0, 3, cap, d, d, d, d, d, d, 16, d) == GSP_ERR_INVALID
    assert lib.gsp_merge_gathered_packed_tree(0, 32, 0, 129, 16, d, d, d, d, d, d, 16, d) == GSP_ERR_INVALID  # 129 * 16 jobs
    torch.cuda.synchronize()
