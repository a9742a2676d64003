"""CPU-side checks of the product's C ABI: the library loads, exports every symbol include/vxb200.h declares,
the Python struct mirrors match the header, and - without a CUDA device - every entry point fails loudly
(there is no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

import voxels_b200
from voxels_b200 import capi

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(REPO, "include", "vxb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vxb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = C.CDLL(voxels_b200.library_path())
    names = declared_symbols()
    assert len(names) >= 15
    for name in names:
        assert hasattr(lib, name), "include/vxb200.h declares %s but libvxb200.so does not export it" % name
    assert sorted(capi.EXPORTED_SYMBOLS) == names, "voxels_b200/capi.py binds a different set than the header declares"


def test_struct_mirrors_match_header_sizes():
    assert capi.RECORD_DTYPE.itemsize == 128 and capi.VERTEX_DTYPE.itemsize == 48
    assert C.sizeof(capi.ResultInfo) == 4 * 4 + 8 * 8 + 20 * 4 + 8 * 4 + 4 + 4
    assert C.sizeof(capi.RegionInfo) == 8 + 2 * 12 * 3 * 4 + 2 * 12 * 4
    assert C.sizeof(capi.ShardBuffers) == 8 * 7 + 4 + 4                                 # vxb_shard_buffers
    assert C.sizeof(capi.NcclId) == 128                                                  # vxb_nccl_id = ncclUniqueId


def test_merge_results_rebases_offsets_and_sorts():
    """capi.merge_results (sharded runs): arenas concatenated in rank order, directory in the reference's block order."""
    import numpy as np

    def fake(level_coord_pairs, nv, ni):
        r = capi.Result.__new__(capi.Result)
        r.n, r.info = 64, None
        r.records = np.zeros(len(level_coord_pairs), capi.RECORD_DTYPE)
        voff = ioff = 0
        for k, (l, c) in enumerate(level_coord_pairs):
            r.records[k]["level"], r.records[k]["coord_id"] = l, c
            r.records[k]["vertex_count"], r.records[k]["index_count"] = nv, ni
            r.records[k]["vertex_offset"], r.records[k]["index_offset"] = voff, ioff
            voff += nv; ioff += ni
        r.verts = np.zeros(voff, capi.VERTEX_DTYPE); r.verts["pos"][:, 0] = np.arange(voff) + 1000 * level_coord_pairs[0][1]
        r.idx = np.arange(ioff, dtype=np.uint32)
        r.tverts = np.zeros(0, capi.VERTEX_DTYPE); r.tidx = np.zeros(0, np.uint32)
        r.stats = np.arange(20, dtype=np.uint32)
        return r

    a, b = fake([(0, 5), (1, 0)], 3, 6), fake([(0, 2), (0, 9)], 2, 3)
    m = capi.merge_results([a, b])
    assert [(int(r["level"]), int(r["coord_id"])) for r in m.records] == [(0, 2), (0, 5), (0, 9), (1, 0)]
    assert len(m.verts) == 10 and len(m.idx) == 18 and np.array_equal(m.stats, 2 * np.arange(20))
    first_b = m.records[0]                                   # rank 1's first block: offsets moved behind rank 0's arenas
    assert first_b["vertex_offset"] == 6 and first_b["index_offset"] == 12
    assert m.verts["pos"][first_b["vertex_offset"], 0] == 2000.0


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(voxels_b200.VxbError) as e:
        voxels_b200.Context(0)
    assert "no CUDA device" in str(e.value) or "CUDA" in str(e.value)


def test_dropin_exports_the_reference_symbols():
    """libvoxels_b200.so must define what the reference's TransVoxelImpl.cpp defines for the public headers."""
    import subprocess
    path = os.path.join(REPO, "voxels_b200", "lib", "libvoxels_b200.so")
    if not os.path.exists(path):
        pytest.skip("drop-in not built (needs the reference headers)")
    out = subprocess.run(["nm", "-D", "--defined-only", "-C", path], capture_output=True, text=True, check=True).stdout
    for sym in ["Voxels::Polygonizer::Polygonizer()", "Voxels::Polygonizer::~Polygonizer()",
                "Voxels::Polygonizer::Execute(Voxels::Grid const&, Voxels::MaterialMap const*, Voxels::Modification*)",
                "Voxels::Modification::Create()", "Voxels::Modification::~Modification()", "Voxels::PolygonSurface::INVALID_ID",
                "InitializeVoxels", "DeinitializeVoxels", "GetBuildVersion", "Voxels::Grid::Create("]:
        assert sym in out, "missing symbol: " + sym


def test_tables_checksum():
    """The generated Transvoxel tables (build/gen, from tests/golden/transvoxel_tables.bin) keep their checksum."""
    text = open(os.path.join(REPO, "build", "gen", "vxb_tables_data.h")).read()
    assert "VXB_TABLES_FNV1A 0x83E0932026BB2FEEull" in text
    assert "Eric Lengyel's Transvoxel Algorithm" in text and "http://www.terathon.com/voxels/" in text


def test_pack_dense_matches_reference_bytes():
    """vxb_pack_dense (host helper of the C ABI) writes exactly the bytes Grid::PackForSave produces (stored digests)."""
    import golden_hash
    import grids
    packs = golden_hash.stored("reference_runs.json")["packs"]
    for name in ("hostile64", "positive_noise32", "plane32"):
        dist, mat, blend = grids.SMALL[name]()
        blob = voxels_b200.pack_dense(dist, mat, blend)
        assert (blob.size, golden_hash._h(blob)) == (packs[name]["bytes"], packs[name]["sha256"]), name


def test_header_is_plain_c(tmp_path):
    """include/vxb200.h is the FFI boundary: it must compile as C99 on its own (no C++/torch types)."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if not gcc:
        pytest.skip("no gcc")
    src = tmp_path / "t.c"
    src.write_text('#include "vxb200.h"\nint main(void) { vxb_result_info i; vxb_block_record r; vxb_shard_buffers x; vxb_nccl_id y; (void)y; (void)i; (void)r; (void)x; return 0; }\n')
    out = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(REPO, "include"), "-fsyntax-only", str(src)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
