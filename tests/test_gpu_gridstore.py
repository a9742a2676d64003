"""Device-resident grid store (SURVEY.md section 8 f1-f3; include/vxb200.h "device-resident grid store") against the
UNMODIFIED reference grid store (src/VoxelGrid.cpp), byte for byte:
  vxb_grid_fill             == Grid::Create(n, n, n, start, step, &surface)      (:79-132)
  vxb_grid_inject_surface   == Grid::InjectSurface  (+ the returned box)           (:388-488)
  vxb_grid_inject_material  == Grid::InjectMaterial (+ the returned box)           (:490-584)
  vxb_grid_pack             == Grid::PackForSave    (CompressBlock + the blob)     (:610-672, :269-315)
and the incremental re-polygonization of device-side edits against the reference's incremental Execute.
The reference's grids and blobs are stored as digests (tests/golden/reference_runs.json, made by
tests/golden/make_golden.py); the incremental test drives the reference itself (oracle/_ref)."""
import numpy as np
import pytest

import compare
import golden_hash
import harness
from voxels_b200 import capi

pytestmark = pytest.mark.gpu


def stored():
    return golden_hash.stored("reference_runs.json")["gridstore"]


def assert_dense_equal(reference, grid, ctx, what=""):
    want = reference.grid_to_dense(grid)
    got = ctx.download_dense()
    for a, b, ch in zip(want, got, ("distance", "material", "blend")):
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            raise AssertionError("%s %s differs at %d voxels, first (z,y,x)=%s: reference %d, device %d"
                                 % (what, ch, len(bad), bad[0], a[tuple(bad[0])], b[tuple(bad[0])]))


def assert_dense_digest(want, ctx, what=""):
    assert golden_hash.input_digest(*ctx.download_dense()) == want, "%s: the device grid differs from the reference's" % what


FILL_CASES = [
    (lambda n: capi.Surface.sphere((n / 2, n / 2, n / 2), 0.3 * n, 2, 17), 64, (0, 0, 0), 1.0),
    (lambda n: capi.Surface.sphere((10.5, 20.25, 30.0), 19.2), 128, (0, 0, 0), 1.0),
    (lambda n: capi.Surface.plane((0.37, 0.61, 0.7), 40.25, 1, 200), 64, (0, 0, 0), 1.0),
    (lambda n: capi.Surface.sphere((3.0, 4.0, 5.0), 6.5), 32, (-2.0, 1.5, 0.25), 0.375),   # the grid samples world space at start + i * step
    (lambda n: capi.Surface.terrain(n), 128, (0, 0, 0), 1.0),
    (lambda n: capi.Surface.terrain(256, origin=(100, 7), seed=99), 64, (0, 0, 96.0), 1.0),
]


@pytest.mark.parametrize("make,n,start,step", FILL_CASES)
def test_fill_equals_reference_constructor(gpu_context, make, n, start, step):
    gpu_context.fill(n, make(n), start, step)
    assert_dense_digest(stored()["fill"][FILL_CASES.index((make, n, start, step))], gpu_context, "fill")


def test_fill_terrain_256_equals_host_generator(gpu_context):
    """the full-size path: device fill vs the reference constructor of the same surface"""
    gpu_context.fill(256, capi.Surface.terrain(256))
    assert_dense_digest(stored()["fill_terrain256"], gpu_context, "fill")


def surface_edits(n, count, seed):
    rng = np.random.RandomState(seed)
    out = []
    for i in range(count):
        r = float(rng.choice([3, 4, 6, 8, 10]))
        if i % 5 == 4:   # fractional centre and odd extents: the reference's float loops (:430-434)
            pos = rng.uniform(8, n - 8, size=3).round(2)
            ext = np.array([2 * r + 3, 2 * r + 5, 2 * r + 1], np.float32)
        else:
            pos = rng.randint(4, n - 4, size=3).astype(np.float32)
            ext = np.full(3, 2 * r + 4, np.float32)
        if i % 7 == 6:   # hanging over the grid edge
            pos[rng.randint(3)] = rng.choice([1.0, n - 2.0])
        out.append((pos.astype(np.float32), ext, capi.Surface.sphere((0, 0, 0), r), i % 3))
    return out


def material_edits(n, count, seed):
    rng = np.random.RandomState(seed)
    out = []
    for i in range(count):
        pos = rng.randint(2, n - 2, size=3).astype(np.float32) if i % 4 else rng.uniform(4, n - 4, size=3).astype(np.float32)
        ext = np.full(3, float(rng.choice([6, 8, 12, 20])), np.float32)
        out.append((pos, ext, int(rng.randint(0, 5)), bool(i % 2)))
    return out


def test_inject_surface_equals_reference(gpu_context):
    n = 64
    gpu_context.fill(n, capi.Surface.terrain(n))
    for i, ((pos, ext, surf, kind), want) in enumerate(zip(surface_edits(n, 40, 5), stored()["inject_surface"])):
        want_box = np.array(want["box"], np.float32)
        got_box = gpu_context.inject_surface(pos, ext, surf, kind)
        assert np.array_equal(want_box, got_box), "edit %d: returned box %s vs %s" % (i, want_box, got_box)
        assert_dense_digest(want["dense"], gpu_context, "edit %d (pos %s ext %s type %d)" % (i, pos, ext, kind))


def test_inject_material_equals_reference(gpu_context):
    n = 64
    gpu_context.fill(n, capi.Surface.terrain(n))
    for i, ((pos, ext, material, add), want) in enumerate(zip(material_edits(n, 30, 11), stored()["inject_material"])):
        want_box = np.array(want["box"], np.float32)
        got_box = gpu_context.inject_material(pos, ext, material, add)
        assert np.array_equal(want_box, got_box)
        assert_dense_digest(want["dense"], gpu_context, "material edit %d" % i)


def pack_input(name, terrain=None):
    """(dist, mat, blend) of a packer test; terrain(n) makes the dense terrain of capi.Surface.terrain(n)."""
    import grids
    if name == "terrain128":
        return terrain(128)
    if name == "zeros32":
        dist = np.zeros((32, 32, 32), np.int8); mat = np.zeros((32, 32, 32), np.uint8); blend = np.full((32, 32, 32), 255, np.uint8)
        dist[:, :, 16:] = 3; dist[5, 5, 5] = -1
        return dist, mat, blend
    return grids.SMALL[name]()


@pytest.mark.parametrize("name", ["terrain128", "hostile64", "noise32", "positive_noise32", "zeros32"])
def test_pack_equals_reference_pack_for_save(gpu_context, name):
    """GPU run-length coding incl. 255-byte run splits, RLE-ineffective (raw) blocks and the BF_Empty flag."""
    def terrain(n):
        gpu_context.fill(n, capi.Surface.terrain(n))
        return gpu_context.download_dense()
    dist, mat, blend = pack_input(name, terrain)
    want = golden_hash.stored("reference_runs.json")["packs"][name]
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"]
    gpu_context.upload_dense(dist, mat, blend)
    got = gpu_context.pack()
    assert len(got) == want["bytes"], "blob size %d vs %d" % (len(got), want["bytes"])
    assert golden_hash._h(got) == want["sha256"], "blob differs from the reference's Grid::PackForSave"
    # and back: the packed form decodes (on the GPU) to the same voxels
    gpu_context.upload_packed(got)
    back = gpu_context.download_dense()
    for a, b in zip((dist, mat, blend), back):
        assert np.array_equal(a, b)


def test_device_edits_then_incremental_polygonize_match_reference(reference, gpu_context):
    """BASELINE configs[4] without the host round trip: edits on the device grid + vxb_polygonize_region, compared with the
    reference's InjectSurface + incremental Execute after every edit (blocks re-created per dirty box, ids, geometry)."""
    n = 128
    s = capi.Surface.terrain(n)
    g = reference.grid_create_builtin(n, s)
    surf, _ = reference.polygonize(g)
    mod = reference.modification_create()
    ctx = gpu_context
    ctx.set_materials(None, None)
    ctx.fill(n, s)
    ctx.polygonize()
    dist0 = reference.grid_to_dense(g)[0]
    rng = np.random.RandomState(3)
    edits = []
    while len(edits) < 25:
        x, y, z = (int(v) for v in rng.randint(16, n - 16, size=3))
        if abs(int(dist0[z, y, x])) >= 4:
            continue
        r = float(rng.choice([4, 6, 8]))
        edits.append((np.array([x, y, z], np.float32), np.full(3, 2 * r + 4, np.float32), capi.Surface.sphere((0, 0, 0), r), 0 if len(edits) % 2 == 0 else 2))
    for i, (pos, ext, sph, kind) in enumerate(edits):
        box = reference.grid_inject_builtin(g, pos, ext, sph, kind)
        s2, _ = reference.polygonize(g, modification=mod, surface=surf, box=box)
        got_box = ctx.inject_surface(pos, ext, sph, kind)
        assert np.array_equal(box, got_box)
        ctx.polygonize_region(got_box[:3], got_box[3:])
        part = ctx.download()
        region = ctx.region_info()
        # the reference's surface after the splice == our previous blocks outside the dirty boxes + the re-created ones
        for l in range(region.levels):
            want = reference.surface_level(surf, l)
            mn, mx = np.array(region.min_dirty[l]), np.array(region.max_dirty[l])
            got = part.level(l)
            # re-created blocks = the tail of the reference's level (erase + append, :443-450, :1293)
            k = len(got.rows)
            tail = harness.LevelDump(want.rows[len(want.rows) - k:], *_tail(want, k))
            problems = compare.level_diff(tail, got, "edit %d L%d" % (i, l))
            assert not problems, "\n".join(problems[:5])
            inside = np.all((want.rows["min"][:len(want.rows) - k] >= mn) & (want.rows["min"][:len(want.rows) - k] < mx), axis=1)
            assert not inside.any(), "edit %d L%d: the reference kept a block inside the dirty box" % (i, l)
    reference.modification_destroy(mod); reference.surface_destroy(surf); reference.grid_destroy(g)


def _tail(level, k):
    r = level.rows
    cut = len(r) - k
    v0 = int(r["nv"][:cut].sum()); i0 = int(r["ni"][:cut].sum()); tv0 = int(r["tnv"][:cut].sum()); ti0 = int(r["tni"][:cut].sum())
    return level.verts[v0:], level.idx[i0:], level.tverts[tv0:], level.tidx[ti0:]
