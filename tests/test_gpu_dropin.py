"""The C++ drop-in (libvoxels_b200.so: Voxels::Polygonizer & co.) driven through the reference's own public API
by the SAME harness source that drives the reference (tests/harness/vxh_capi.cpp), and compared with it."""
import os

import numpy as np
import pytest

import compare
import grids
import harness

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dropin():
    if not os.path.exists(harness.B200_LIB):
        pytest.skip("build/libvxh_b200.so not built (the drop-in links the reference's grid store: build() with a reference checkout)")
    return harness.load(harness.B200_LIB)


def both(reference, dropin, make_grid, **kw):
    out = []
    for lib in (reference, dropin):
        g = make_grid(lib)
        s, sec = lib.polygonize(g, **kw)
        assert s, "Execute returned nullptr (%s)" % lib.path
        levels = [lib.surface_level(s, l) for l in range(lib.surface_levels(s))]
        out.append((levels, lib.surface_stats(s), lib.surface_extents(s), lib.L.vxh_surface_cache_bytes(s), lib.L.vxh_surface_polygon_bytes(s)))
        lib.surface_destroy(s)
        lib.grid_destroy(g)
    return out


def assert_same(a, b):
    (la, sa, ea, ca, pa), (lb, sb, eb, cb, pb) = a, b
    assert len(la) == len(lb)
    problems = []
    for l, (x, y) in enumerate(zip(la, lb)):
        problems += compare.level_diff(x, y, "L%d" % l)
    assert not problems, "\n".join(problems[:10])
    assert np.array_equal(sa, sb), "statistics differ: %s vs %s" % (sa, sb)
    assert np.array_equal(ea, eb)
    assert ca == cb, "GetCacheSizeBytes %d vs %d" % (ca, cb)
    assert pa == pb, "GetPolygonDataSizeBytes %d vs %d" % (pa, pb)


def test_client_flow_sphere64(reference, dropin):
    """BASELINE config 1: Grid::Create(64,64,64,...,&sphere) -> Polygonizer::Execute, exactly as a client would."""
    a, b = both(reference, dropin, lambda lib: lib.grid_sphere(64, (32, 32, 32), 19.2))
    assert_same(a, b)
    assert a[1][0] == 73 and a[1][2] == 9096  # SURVEY.md 8(d) config 1 anchors: blocks calculated, non-trivial cells
    assert len(a[0][0].verts) == 8832 and len(a[0][0].idx) == 41496


@pytest.mark.parametrize("name", ["hostile64", "plane32", "noise32"])
def test_dense_grids(reference, dropin, name):
    dist, mat, blend = grids.SMALL[name]()
    a, b = both(reference, dropin, lambda lib: lib.grid_from_dense(dist, mat, blend))
    assert_same(a, b)


def test_unmapped_material_logs_per_vertex(reference, dropin):
    dist, mat, blend = grids.SMALL["hostile64"]()
    valid = np.ones(256, np.uint8); valid[2] = 0
    before = [lib.L.vxh_error_logs() for lib in (reference, dropin)]
    a, b = both(reference, dropin, lambda lib: lib.grid_from_dense(dist, mat, blend), valid_mask=valid)
    assert_same(a, b)
    after = [lib.L.vxh_error_logs() for lib in (reference, dropin)]
    assert after[0] - before[0] == after[1] - before[1] > 0  # one LS_Error per vertex with the unmapped material


def _edit_sequence(n, count, seed=42):
    """BASELINE config 5 shape: seeded sphere add/subtract edits with integer centres and even extents."""
    rng = np.random.RandomState(seed)
    edits = []
    for i in range(count):
        r = int(rng.choice([4, 6, 8, 10]))
        pos = [int(v) for v in rng.randint(24, n - 24, size=3)]
        pos[2] = int(n // 2 + rng.randint(-10, 10))  # near the terrain surface
        edits.append((pos, float(r), float(2 * r + 4), harness.IT_ADD if i % 2 == 0 else harness.IT_SUBTRACT))
    return edits


@pytest.mark.parametrize("name,n,count", [("hostile", 64, 12), ("terrain", 128, 20)])
def test_incremental_edits_match_reference(reference, dropin, name, n, count):
    """Execute(grid, materials, modification) after Grid::InjectSurface: the drop-in must follow the reference's
    INCREMENTAL behaviour (stale consistency bits, vote-only cache overwrites, id continuation, erase + append order),
    which is not the same as a fresh polygonization (SURVEY.md 8 a9)."""
    if name == "hostile":
        import gridgen
        dist, mat, blend = gridgen.hostile(n, seed=3)
    else:
        from voxels_b200 import synth
        dist, mat, blend = (t.numpy() for t in synth.terrain(n))
    state = []
    for lib in (reference, dropin):
        g = lib.grid_from_dense(dist, mat, blend)
        s, _ = lib.polygonize(g)
        state.append([lib, g, s, lib.modification_create()])
    for step, (pos, radius, extent, kind) in enumerate(_edit_sequence(n, count)):
        dumps = []
        for st in state:
            lib, g, s, mod = st
            box = lib.grid_inject_sphere(g, pos, radius, extent, kind)
            s2, _ = lib.polygonize(g, modification=mod, surface=s, box=box)
            assert s2 == s, "Execute must return the surface it was given"
            dumps.append(([lib.surface_level(s, l) for l in range(lib.surface_levels(s))], lib.surface_stats(s), lib.modification_blocks(mod), box))
        (la, sa, ma, ba), (lb, sb, mb, bb) = dumps
        assert np.array_equal(ba, bb)
        problems = []
        for l, (x, y) in enumerate(zip(la, lb)):
            problems += compare.level_diff(x, y, "edit %d L%d" % (step, l))
        assert not problems, "\n".join(problems[:10])
        assert np.array_equal(sa, sb), "edit %d statistics: %s vs %s" % (step, sa, sb)
        assert np.array_equal(ma, mb), "edit %d ModifiedBlocks differ" % step
    for lib, g, s, mod in state:
        lib.modification_destroy(mod); lib.surface_destroy(s); lib.grid_destroy(g)


def test_config5_terrain_512_1000_edits(reference, dropin):
    """BASELINE configs[4] as written: 512^3 terrain, 1000 seeded sphere add/subtract edits near the surface, incremental
    re-polygonization after each; the two surfaces (all levels, statistics, ModifiedBlocks) are compared every 100 edits."""
    import sys
    import torch
    from voxels_b200 import synth
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import bench_edits
    n = 512
    dist, mat, blend = (t.cpu().numpy() for t in synth.terrain(n, "cuda:0" if torch.cuda.is_available() else "cpu"))
    edits = bench_edits.edit_sequence(n, 1000, dist)
    state = []
    for lib in (reference, dropin):
        g = lib.grid_from_dense(dist, mat, blend)
        s, _ = lib.polygonize(g)
        state.append([lib, g, s, lib.modification_create()])
    for step, (pos, radius, extent, kind) in enumerate(edits):
        boxes = []
        for lib, g, s, mod in state:
            box = lib.grid_inject_sphere(g, pos, radius, extent, kind)
            s2, _ = lib.polygonize(g, modification=mod, surface=s, box=box)
            assert s2 == s
            boxes.append(box)
        assert np.array_equal(boxes[0], boxes[1])
        if (step + 1) % 100 == 0:
            (la, ga, sa, ma), (lb, gb, sb, mb) = state
            problems = []
            for l in range(la.surface_levels(sa)):
                problems += compare.level_diff(la.surface_level(sa, l), lb.surface_level(sb, l), "edit %d L%d" % (step, l))
            assert not problems, "\n".join(problems[:10])
            assert np.array_equal(la.surface_stats(sa), lb.surface_stats(sb))
            assert np.array_equal(la.modification_blocks(ma), lb.modification_blocks(mb))
    for lib, g, s, mod in state:
        lib.modification_destroy(mod); lib.surface_destroy(s); lib.grid_destroy(g)
