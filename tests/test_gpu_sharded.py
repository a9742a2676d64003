"""Sharded runs (include/vxb200.h: vxb_polygonize_sharded, vxb_shard_*, vxb_cube_*; SURVEY.md section 8e) on ONE GPU.

`world` contexts of one process play the ranks: each scans its own z-pieces, the block-info all-gather is a device
copy, the page exchange goes through the same peer stores a real run uses (the "peer" buffers live on the same device),
and the merged result must be bit-identical to the unsharded run - and thus to the reference.  The cube test backs every
piece with its own cuMemCreate allocation and maps the "peers'" pieces through exported file descriptors, exactly what
the ranks of a torchrun job do with each other's HBM."""
import os

import numpy as np
import pytest

import compare
import grids

pytestmark = pytest.mark.gpu


def _view(ptr, nbytes):
    import torch
    from voxels_b200 import capi
    return torch.as_tensor(capi.DevicePointer(ptr, nbytes), device=torch.device("cuda", 0))


def configure_virtual_ranks(contexts, group_planes=0):
    world = len(contexts)
    for r, c in enumerate(contexts):
        c.shard_configure(r, world, group_planes)
    bufs = [c.shard_buffers() for c in contexts]
    for r, c in enumerate(contexts):
        for p in range(world):
            if p != r:
                c.shard_set_peer(p, bufs[p].pages, bufs[p].valid)
    return bufs


def run_virtual_ranks(contexts, bufs, flags=0):
    """contexts[r] already sees the whole grid and is configured.  Returns (merged result, per-rank infos)."""
    import torch
    from voxels_b200 import capi
    world = len(contexts)
    for attempt in range(4):
        for c in contexts:
            c.polygonize_sharded(0, flags)
        torch.cuda.synchronize()
        # exchange 0: all-gather of the per-block info (rank r's chunk = bytes [r, r+1) * chunk_bytes)
        chunk = bufs[0].chunk_bytes
        views = [_view(b.block_info, b.block_info_bytes) for b in bufs]
        for src in range(world):
            for dst in range(world):
                if src != dst:
                    views[dst][src * chunk:(src + 1) * chunk].copy_(views[src][src * chunk:(src + 1) * chunk])
        torch.cuda.synchronize()
        for c in contexts:
            c.polygonize_sharded(1, flags)
        torch.cuda.synchronize()  # exchange 1: the pages were stored into the peers' buffers by phase 1
        rcs = [c.polygonize_sharded(2, flags) for c in contexts]
        if not any(rcs):
            return capi.merge_results([c.download() for c in contexts]), [c.info() for c in contexts]
    raise AssertionError("arenas kept overflowing")


def assert_same(a, b, levels):
    problems = []
    for l in range(levels):
        problems += compare.level_diff(a.level(l), b.level(l), "L%d" % l)
    if not np.array_equal(a.stats, b.stats):
        problems.append("stats differ: %s vs %s" % (a.stats, b.stats))
    assert not problems, "\n".join(problems[:10])


@pytest.mark.parametrize("name,world,group", [("hostile128", 2, 0), ("hostile128", 4, 32), ("hostile128", 2, 32), ("sphere128", 2, 0),
                                              ("noise64", 2, 0), ("hostile64", 2, 0), ("hostile128", 1, 0), ("sphere128", 4, 0)])
def test_virtual_ranks_equal_single_run(gpu_context, name, world, group):
    import voxels_b200
    dist, mat, blend = (grids.MEDIUM.get(name) or grids.SMALL[name])()
    n = dist.shape[0]
    gpu_context.set_materials(None, None)
    gpu_context.upload_dense(dist, mat, blend)
    info = gpu_context.polygonize()
    single = gpu_context.download()
    d, m, b = gpu_context.device_pointers()
    contexts = [voxels_b200.Context(0) for _ in range(world)]
    try:
        for c in contexts:
            c.set_device_grid(n, d, m, b)
        bufs = configure_virtual_ranks(contexts, group)
        merged, infos = run_virtual_ranks(contexts, bufs)
        assert_same(single, merged, info.levels_total)
        # every block exactly once, ids are the full-run ids
        assert np.array_equal(single.records["id"], merged.records["id"])
        if world > 1 and name != "noise64":
            assert sum(1 for i in infos if i.block_count) > 1, "the work was not split"
    finally:
        for c in contexts:
            c.close()


def test_sharded_against_reference(gpu_context):
    import golden_hash
    import voxels_b200
    dist, mat, blend = grids.MEDIUM["hostile128"]()
    want = golden_hash.reference_run("hostile128")
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"]
    gpu_context.upload_dense(dist, mat, blend)
    d, m, b = gpu_context.device_pointers()
    contexts = [voxels_b200.Context(0) for _ in range(4)]
    try:
        for c in contexts:
            c.set_device_grid(128, d, m, b)
        bufs = configure_virtual_ranks(contexts)
        merged, _ = run_virtual_ranks(contexts, bufs)
        problems = golden_hash.run_problems(want, merged, len(want["levels"]))
        assert not problems, "\n".join(problems[:10])
    finally:
        for c in contexts:
            c.close()


def _terrain(n):
    import torch
    from voxels_b200 import synth
    dev = torch.device("cuda", 0)
    return synth.terrain(n, dev)


def test_sharded_terrain_512_balance_and_parity(gpu_context):
    """512^3 terrain (surface in a few z-layers) over 4 and 8 virtual ranks: bit-identical to the single run, and the
    work split is by blocks, not by where the data lives: no rank gets more than 1.35x its fair share of the vertices."""
    import torch
    import voxels_b200
    n = 512
    dist, mat, blend = _terrain(n)
    torch.cuda.synchronize()
    gpu_context.set_materials(None, None)
    gpu_context.set_device_grid(n, dist.data_ptr(), mat.data_ptr(), blend.data_ptr(), keep=(dist, mat, blend))
    info = gpu_context.polygonize()
    single = gpu_context.download()
    for world in (4, 8):
        contexts = [voxels_b200.Context(0) for _ in range(world)]
        try:
            for c in contexts:
                c.set_device_grid(n, dist.data_ptr(), mat.data_ptr(), blend.data_ptr())
            bufs = configure_virtual_ranks(contexts, 32)
            merged, infos = run_virtual_ranks(contexts, bufs)
            assert_same(single, merged, info.levels_total)
            share = np.array([i.vertex_total for i in infos], np.float64)
            assert share.max() <= 1.35 * share.sum() / world, share
        finally:
            for c in contexts:
                c.close()


@pytest.mark.parametrize("world,group", [(1, 0), (2, 0), (4, 0), (2, 32), (4, 32)])
def test_cube_of_mapped_pieces(gpu_context, world, group):
    """The VMM cube: one virtual range per volume, every piece its own physical allocation, peers imported by descriptor."""
    import torch
    import voxels_b200
    from voxels_b200.dist import owned_pieces
    n = 256
    dev = torch.device("cuda", 0)
    dist, mat, blend = _terrain(n)
    gpu_context.set_materials(None, None)
    gpu_context.set_device_grid(n, dist.data_ptr(), mat.data_ptr(), blend.data_ptr(), keep=(dist, mat, blend))
    info = gpu_context.polygonize()
    single = gpu_context.download()
    contexts = [voxels_b200.Context(0) for _ in range(world)]
    g = group or n // world
    try:
        for r, c in enumerate(contexts):
            c.cube_create(n, r, world, group)
        channels = contexts[0].cube_info()[1]
        for r, c in enumerate(contexts):
            for p, z0, z1 in owned_pieces(n, r, world, g):
                for ch in range(channels):
                    fd = c.cube_export(ch, p)
                    for q, peer in enumerate(contexts):
                        if q != r:
                            peer.cube_import(ch, p, fd)
                    os.close(fd)
                pd, pm, pbl, size = c.cube_piece(p)
                assert size == n * n * (z1 - z0)
                for ptr, src in ((pd, dist), (pm, mat), (pbl, blend)):
                    _view(ptr, size).copy_(src[z0:z1].reshape(-1).view(torch.uint8))
        torch.cuda.synchronize()
        # the page buffers: exported / imported like the pieces
        for r, c in enumerate(contexts):
            c.shard_configure(r, world, group)
        for r, c in enumerate(contexts):
            if world > 1:
                fd = c.shard_export()
                for q, peer in enumerate(contexts):
                    if q != r:
                        peer.shard_import(r, fd)
                os.close(fd)
        bufs = [c.shard_buffers() for c in contexts]
        merged, _ = run_virtual_ranks(contexts, bufs)
        assert_same(single, merged, info.levels_total)
    finally:
        for c in contexts:
            c.close()
