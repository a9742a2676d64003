"""GPU parity: the CUDA path (through the C ABI, include/vxb200.h) against the unmodified reference.

Bit-exact: block ids/order/corners, counts, indices, transition indices, texture bytes, flag bits,
positions, statistics.  Normals: <= 1e-5 (contract of BASELINE.json's north_star), 0 ULP expected - and found, so the
reference's output is stored as digests of every field (tests/golden, made by tests/golden/make_golden.py)."""
import numpy as np
import pytest

import compare
import golden_hash
import grids

pytestmark = pytest.mark.gpu


def run_both(reference_run, ctx, dist, mat, blend, table=None, valid=None, max_levels=0, flags=0):
    """The CUDA path on the given input against the stored run of the reference (golden_hash.reference_run) on it."""
    want = golden_hash.reference_run(reference_run)
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"], "input differs from the one the reference ran on"
    ctx.set_materials(table, valid)
    ctx.upload_dense(dist, mat, blend)
    info = ctx.polygonize(max_levels, flags)
    res = ctx.download()
    levels = len(want["levels"])
    assert info.levels_total == levels
    ncmp = levels if max_levels == 0 else min(levels, max_levels)
    return golden_hash.run_problems(want, res, ncmp, stats=max_levels == 0), res


def material_table_and_valid_ids():
    table = (np.arange(256 * 6) * 7 % 251).astype(np.uint8)
    valid = np.ones(256, np.uint8); valid[1] = 0  # GetMaterial(1) -> nullptr: textures stay zero (TransVoxelImpl.cpp:1364-1368)
    return table, valid


@pytest.mark.parametrize("name", sorted(grids.SMALL))
def test_small_grids_all_levels(gpu_context, name):
    dist, mat, blend = grids.SMALL[name]()
    problems, res = run_both(name, gpu_context, dist, mat, blend)
    assert not problems, "\n".join(problems[:10])


@pytest.mark.parametrize("name", sorted(grids.MEDIUM))
def test_medium_grids_all_levels(gpu_context, name):
    dist, mat, blend = grids.MEDIUM[name]()
    problems, res = run_both(name, gpu_context, dist, mat, blend)
    assert not problems, "\n".join(problems[:10])


def test_material_table_and_invalid_ids(gpu_context):
    dist, mat, blend = grids.SMALL["hostile64"]()
    table, valid = material_table_and_valid_ids()
    problems, res = run_both("hostile64_material_table", gpu_context, dist, mat, blend, table=table, valid=valid)
    assert not problems, "\n".join(problems[:10])


def test_level0_only_regular_cells(gpu_context):
    """BASELINE config 2 shape: single LOD, regular cells only."""
    import voxels_b200
    dist, mat, blend = grids.MEDIUM["hostile128"]()
    problems, res = run_both("hostile128", gpu_context, dist, mat, blend, max_levels=1, flags=voxels_b200.FLAG_NO_TRANSITIONS)
    assert not problems, "\n".join(problems[:10])


def test_block_upload_equals_dense_upload(gpu_context):
    dist, mat, blend = grids.SMALL["hostile64"]()
    n = dist.shape[0]; nb = n // 16

    def to_blocks(a):
        return np.ascontiguousarray(a.reshape(nb, 16, nb, 16, nb, 16).transpose(0, 2, 4, 1, 3, 5)).reshape(-1)

    gpu_context.set_materials(None, None)
    gpu_context.upload_dense(dist, mat, blend)
    gpu_context.polygonize()
    a = gpu_context.download()
    gpu_context.upload_blocks(n, to_blocks(dist), to_blocks(mat), to_blocks(blend))
    gpu_context.polygonize()
    b = gpu_context.download()
    for l in range(a.info.levels_total):
        assert not compare.level_diff(a.level(l), b.level(l), "L%d" % l)


def test_packed_upload_equals_dense_upload(gpu_context):
    """vxb_grid_upload_packed: the reference's own PackForSave bytes, run-length decoded on the GPU."""
    import voxels_b200
    packs = golden_hash.stored("reference_runs.json")["packs"]
    for name in ("hostile64", "positive_noise32", "noise32"):  # incl. RLE-ineffective (raw) blocks
        dist, mat, blend = grids.SMALL[name]()
        blob = voxels_b200.pack_dense(dist, mat, blend)
        assert golden_hash._h(blob) == packs[name]["sha256"], "host packer differs from Grid::PackForSave"
        gpu_context.set_materials(None, None)
        gpu_context.upload_dense(dist, mat, blend)
        gpu_context.polygonize()
        a = gpu_context.download()
        gpu_context.upload_packed(blob)
        gpu_context.polygonize()
        b = gpu_context.download()
        for l in range(a.info.levels_total):
            assert not compare.level_diff(a.level(l), b.level(l), "%s L%d" % (name, l))
        assert np.array_equal(a.stats, b.stats)


def test_arena_growth_retry(gpu_context):
    """Tiny initial arenas: the run must detect the overflow, grow and still match."""
    import voxels_b200
    ctx = voxels_b200.Context(0)
    try:
        ctx.set_capacity(1024, 1024, 64, 64)
        dist, mat, blend = grids.SMALL["hostile64"]()
        problems, res = run_both("hostile64", ctx, dist, mat, blend)
        assert not problems, "\n".join(problems[:10])
    finally:
        ctx.close()


def test_repeatable(gpu_context):
    dist, mat, blend = grids.SMALL["hostile64"]()
    gpu_context.set_materials(None, None)
    gpu_context.upload_dense(dist, mat, blend)
    gpu_context.polygonize(); a = gpu_context.download()
    gpu_context.polygonize(); b = gpu_context.download()
    for l in range(a.info.levels_total):
        assert not compare.level_diff(a.level(l), b.level(l), "L%d" % l)
    assert np.array_equal(a.stats, b.stats)


# ---- committed digests of the reference's output (tests/golden): no reference needed at run time ----------------
import json
import os

import golden_hash


def _golden():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_hashes.json")) as f:
        return json.load(f)["grids"]


@pytest.mark.parametrize("name", sorted(list(grids.SMALL) + list(grids.MEDIUM)))
def test_matches_golden_digests(gpu_context, name):
    dist, mat, blend = (grids.SMALL.get(name) or grids.MEDIUM[name])()
    want = _golden()[name]
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"]
    gpu_context.set_materials(None, None)
    gpu_context.upload_dense(dist, mat, blend)
    info = gpu_context.polygonize()
    res = gpu_context.download()
    assert [int(v) for v in res.stats] == want["stats"]
    assert info.levels_total == len(want["levels"])
    for l, w in enumerate(want["levels"]):
        got = golden_hash.level_digests(res.level(l))
        assert got["counts"] == w["counts"], "level %d counts" % l
        assert got["exact"] == w["exact"], "level %d bit-exact fields" % l
        assert got["normals"] == w["normals"], "level %d normals differ in bits (contract allows 1e-5, 0 ULP expected)" % l


def test_terrain_256_against_reference(gpu_context):
    from voxels_b200 import synth
    dist, mat, blend = (t.numpy() for t in synth.terrain(256))
    problems, res = run_both("terrain256", gpu_context, dist, mat, blend)
    assert not problems, "\n".join(problems[:10])


def test_full_size_properties_1024(gpu_context):
    """BASELINE full size (1024^3 terrain, all levels): size-independent properties, no oracle needed."""
    import torch
    from voxels_b200 import synth
    n = 1024
    dist, mat, blend = synth.terrain(n, "cuda:0")
    torch.cuda.synchronize()
    gpu_context.set_materials(None, None)
    gpu_context.set_device_grid(n, dist.data_ptr(), mat.data_ptr(), blend.data_ptr(), keep=(dist, mat, blend))
    info = gpu_context.polygonize()
    res = gpu_context.download()
    recs = res.records
    assert info.levels_total == 7 and info.block_count == len(recs) > 1000
    # directory is in the reference's order: level, then z,y,x
    key = recs["level"].astype(np.int64) * (1 << 32) + recs["coord_id"]
    assert np.all(np.diff(key) > 0)
    # ids follow GenerateBlockListForLevel: running counter over all blocks of all lower levels + coord id
    base = np.cumsum([0] + [((n // 16) >> l) ** 3 for l in range(7)])
    assert np.array_equal(recs["id"], base[recs["level"]] + recs["coord_id"])
    st = res.stats
    assert st[0] == base[7]                                  # BlocksCalculated = every block of every level
    assert st[4:].sum() == st[2]                             # per-class histogram sums to NonTrivialCells
    assert (int(st[1]) + int(st[2])) % 4096 == 0            # whole blocks were classified
    assert info.vertex_total == recs["vertex_count"].sum() and info.index_total == recs["index_count"].sum()
    # every index addresses a vertex of its own block; every kept triangle passes the reference's degenerate test
    rng = np.random.RandomState(1)
    for i in rng.choice(len(recs), 200, replace=False):
        r = recs[i]
        v = res.verts[r["vertex_offset"]:r["vertex_offset"] + r["vertex_count"]]
        ix = res.idx[r["index_offset"]:r["index_offset"] + r["index_count"]]
        assert len(ix) % 3 == 0 and (len(ix) == 0 or ix.max() < len(v))
        m = 16 << int(r["level"]); nb = n // m; c = int(r["coord_id"])
        lo = np.array([c % nb, c // (nb * nb), (c // nb) % nb], np.float32) * m   # output axes: (x, z, y)
        assert np.all(v["pos"] >= lo - 1e-3) and np.all(v["pos"] <= lo + m + 1e-3)
        p = (v["pos"][:, [0, 2, 1]] * np.float32(256)).astype(np.float32)
        a, b, cc = p[ix[0::3]], p[ix[1::3]], p[ix[2::3]]
        cr = np.cross((b - a).astype(np.float32), (cc - a).astype(np.float32)).astype(np.float64)
        assert np.all((cr ** 2).sum(axis=1) >= 1.1920928955078125e-07 * 0.5)
        nl = np.linalg.norm(v["nrm"].astype(np.float64), axis=1)
        assert np.all((np.abs(nl - 1) < 1e-5) | (nl == 0))
        for f in range(6):
            tv, ti = int(r["trans_vertex_count"][f]), int(r["trans_index_count"][f])
            tix = res.tidx[r["trans_index_offset"][f]:r["trans_index_offset"][f] + ti]
            assert ti % 3 == 0 and (ti == 0 or tix.max() < tv)
    # idempotence: a second run gives the same bytes
    gpu_context.polygonize()
    res2 = gpu_context.download()
    for l in range(7):
        assert golden_hash.level_digests(res.level(l)) == golden_hash.level_digests(res2.level(l))
    # level 0 alone (BASELINE config 2 shape) equals level 0 of the full run
    import voxels_b200
    gpu_context.polygonize(1, voxels_b200.FLAG_NO_TRANSITIONS)
    res3 = gpu_context.download()
    assert golden_hash.level_digests(res.level(0)) == golden_hash.level_digests(res3.level(0))


# ---- BASELINE sizes against the unmodified reference (stored runs), end to end (TransVoxelImpl.cpp:468-538) ------
def _terrain_numpy(n):
    """On the CPU: the bytes the stored reference runs were made from (torch's CUDA kernels round the terrain's float
    math differently in a few voxels)."""
    from voxels_b200 import synth
    return tuple(t.numpy() for t in synth.terrain(n))


def test_config2_terrain_512_level0_regular_cells_against_reference(gpu_context):
    """BASELINE configs[1]: 512^3 Perlin terrain, single LOD, regular cells only - level 0 bit-exact vs the reference."""
    import voxels_b200
    dist, mat, blend = _terrain_numpy(512)
    problems, res = run_both("terrain512", gpu_context, dist, mat, blend, max_levels=1, flags=voxels_b200.FLAG_NO_TRANSITIONS)
    assert not problems, "\n".join(problems[:10])
    assert len(res.records) > 1000


def test_config2_terrain_512_all_levels_against_reference(gpu_context):
    dist, mat, blend = _terrain_numpy(512)
    problems, res = run_both("terrain512", gpu_context, dist, mat, blend)
    assert not problems, "\n".join(problems[:10])


def test_config3_terrain_1024_levels_0_to_3_with_transitions_against_reference(gpu_context):
    """BASELINE configs[2]: 1024^3 terrain, 4 LOD levels + transition cells.  The reference always computes all 7
    levels; levels 0-3 (level-3 transitions included: 3 is not the last level) are compared bit-exactly."""
    dist, mat, blend = _terrain_numpy(1024)
    problems, res = run_both("terrain1024", gpu_context, dist, mat, blend, max_levels=4)
    assert not problems, "\n".join(problems[:10])
    assert res.info.levels_computed == 4 and res.info.trans_vertex_total > 0


def test_config3_terrain_1024_all_levels_against_reference(gpu_context):
    """The bench workload itself (1024^3, all 7 levels + transitions): every block, vertex, index and the statistics."""
    dist, mat, blend = _terrain_numpy(1024)
    problems, res = run_both("terrain1024", gpu_context, dist, mat, blend)
    assert not problems, "\n".join(problems[:10])


def test_packed_upload_rejects_malformed_blobs():
    """A blob whose size table, length or per-block flags are inconsistent must fail with an argument error (never read out
    of bounds, never leave a half-decoded grid behind): the flags words are checked by the decoding kernel itself."""
    import voxels_b200
    from voxels_b200 import capi
    dist, mat, blend = grids.SMALL["hostile64"]()
    good = voxels_b200.pack_dense(dist, mat, blend).copy()
    ctx = voxels_b200.Context(0)
    try:
        ctx.upload_packed(good)
        nb = 4; table = 16; data0 = 16 + nb ** 3 * 12
        sizes = good[table:data0].view(np.uint32).reshape(-1, 3)
        cases = {}
        b = good.copy(); b[table:table + 4].view(np.uint32)[0] = 5000; cases["size > 4096 in the table"] = b
        cases["truncated"] = good[:len(good) - 100].copy()
        b = good.copy(); b[data0:data0 + 4].view(np.uint32)[0] |= 2; cases["raw flag on a run-length coded channel"] = b   # block 0: BF_DistanceUncompressed but size < 4096
        assert sizes[0, 0] < 4096
        b = good.copy(); b[data0 + 4] = (int(b[data0 + 4]) + 1) & 0xFF; cases["run lengths that do not add up to 4096"] = b   # first run of block 0's distance channel
        for what, blob in cases.items():
            with pytest.raises(capi.VxbError):
                ctx.upload_packed(blob)
            with pytest.raises(capi.VxbError):   # no grid after a failed upload
                ctx.polygonize()
        ctx.upload_packed(good)                  # and the context still works
        ctx.polygonize()
    finally:
        ctx.close()


def test_streamed_packed_upload_and_split_download():
    """vxb_grid_upload_packed_streamed with a producer that writes each slab only when asked equals the plain packed upload,
    every layer is asked for exactly once in ascending order; vxb_result_download_begin/_end equals vxb_result_download."""
    import voxels_b200
    from voxels_b200 import capi
    dist, mat, blend = grids.MEDIUM["hostile128"]()
    n = 128; nb = n // 16
    good = voxels_b200.pack_dense(dist, mat, blend).copy()
    head = 16 + nb ** 3 * 12
    sizes = good[16:head].view(np.uint32).reshape(-1, 3).astype(np.int64)
    offsets = head + np.concatenate([[0], np.cumsum(4 + sizes.sum(axis=1))])
    ctx = voxels_b200.Context(0)
    try:
        ctx.upload_packed(good)
        ctx.polygonize()
        want = ctx.download()
        want_dense = ctx.download_dense()
        blob = good.copy()
        blob[head:] = 0xEE                      # no block data yet
        asked = []

        def produce(l0, l1):
            asked.append((l0, l1))
            a, b = offsets[l0 * nb * nb], offsets[l1 * nb * nb]
            blob[a:b] = good[a:b]
        ctx.upload_packed_streamed(blob, produce)
        assert asked and asked[0][0] == 0 and asked[-1][1] == nb and all(asked[i][1] == asked[i + 1][0] for i in range(len(asked) - 1))
        got_dense = ctx.download_dense()
        for a, b in zip(want_dense, got_dense):
            assert np.array_equal(a, b)
        info = ctx.polygonize()
        res = ctx.download_begin()
        for f in ("level", "coord_id", "id", "vertex_count", "index_count"):   # the directory is there before the arenas (offsets differ run to run)
            assert np.array_equal(res.records[f], want.records[f]), f
        with pytest.raises(capi.VxbError):                     # no run while a download is open
            ctx.polygonize()
        ctx.download_end()
        problems = []
        for l in range(info.levels_total):
            problems += compare.level_diff(want.level(l), res.level(l), "L%d" % l)
        assert not problems, "\n".join(problems[:10])
        with pytest.raises(capi.VxbError):
            ctx.download_end()
    finally:
        ctx.close()
