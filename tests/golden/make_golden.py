#!/usr/bin/env python
"""Regenerates tests/golden/reference_hashes.json and tests/golden/reference_runs.json FROM THE UNMODIFIED REFERENCE
(oracle/_ref, built by `make -C oracle ref` from a checkout of the reference).  The reference ships no golden vectors or
tests of its own (SURVEY.md section 4), so these are outputs of the reference itself on the seeded inputs the tests use,
reduced to SHA-256 digests; the tests check the CUDA path and the CPU restatement against them without the reference.

    python tests/golden/make_golden.py

reference_hashes.json: Polygonizer::Execute on the named grids of tests/grids.py.
reference_runs.json:   runs:        Execute on the other inputs of the parity tests (material table, synth terrains)
                       packs:       Grid::PackForSave of the packer tests' grids
                       empty_flags: the reference's BF_Empty block flags of tests/grids.py's small grids
                       gridstore:   Grid::Create / InjectSurface / InjectMaterial of tests/test_gpu_gridstore.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import golden_hash  # noqa: E402
import grids  # noqa: E402
import harness  # noqa: E402


def run_entry(ref, dist, mat, blend, table=None, valid=None):
    g = ref.grid_from_dense(dist, mat, blend)
    s, _ = ref.polygonize(g, material_table=table, valid_mask=valid)
    entry = {"input_sha256": golden_hash.input_digest(dist, mat, blend), "stats": [int(v) for v in ref.surface_stats(s)], "levels": []}
    for l in range(ref.surface_levels(s)):
        entry["levels"].append(golden_hash.level_digests(ref.surface_level(s, l)))
    ref.surface_destroy(s); ref.grid_destroy(g)
    return entry


def sha(a):
    return golden_hash._h(a)


def reference_hashes(ref):
    out = {"_comment": "SHA-256 of the reference's own output (see make_golden.py); regenerate, never edit", "grids": {}}
    for name in sorted(list(grids.SMALL) + list(grids.MEDIUM)):
        entry = run_entry(ref, *(grids.SMALL.get(name) or grids.MEDIUM[name])())
        out["grids"][name] = entry
        print(name, entry["stats"][:4], [lv["counts"] for lv in entry["levels"]])
    return out


def reference_runs(ref):
    import test_gpu_gridstore as gs
    import test_gpu_parity as gp
    from voxels_b200 import capi, synth
    out = {"_comment": "SHA-256 of the reference's own output (see make_golden.py); regenerate, never edit",
           "runs": {}, "packs": {}, "empty_flags": {}, "gridstore": {}}
    runs = out["runs"]
    runs["hostile64_material_table"] = run_entry(ref, *grids.SMALL["hostile64"](), *gp.material_table_and_valid_ids())
    for n in (64, 256, 512, 1024):
        dist, mat, blend = (t.numpy() for t in synth.terrain(n))
        runs["terrain%d" % n] = run_entry(ref, dist, mat, blend)
        print("terrain%d" % n, runs["terrain%d" % n]["stats"][:4])
        del dist, mat, blend

    for name in ("hostile64", "positive_noise32", "noise32", "plane32", "zeros32", "terrain128"):
        dist, mat, blend = gs.pack_input(name, lambda n: ref.builtin_dense(n, capi.Surface.terrain(n)))
        g = ref.grid_from_dense(dist, mat, blend)
        blob = ref.grid_pack(g)
        out["packs"][name] = {"input_sha256": golden_hash.input_digest(dist, mat, blend), "bytes": int(blob.size), "sha256": sha(blob)}
        if name in grids.SMALL:
            out["empty_flags"][name] = sha(ref.grid_empty_flags(g))
        ref.grid_destroy(g)
    for name in grids.SMALL:
        if name not in out["empty_flags"]:
            g = ref.grid_from_dense(*grids.SMALL[name]())
            out["empty_flags"][name] = sha(ref.grid_empty_flags(g))
            ref.grid_destroy(g)

    st = out["gridstore"]
    st["fill"] = []
    for make, n, start, step in gs.FILL_CASES:
        g = ref.grid_create_builtin(n, make(n), start, step)
        st["fill"].append(golden_hash.input_digest(*ref.grid_to_dense(g)))
        ref.grid_destroy(g)
    g = ref.grid_create_builtin(256, capi.Surface.terrain(256))
    st["fill_terrain256"] = golden_hash.input_digest(*ref.grid_to_dense(g))
    ref.grid_destroy(g)
    n = 64
    g = ref.grid_create_builtin(n, capi.Surface.terrain(n))
    st["inject_surface"] = []
    for pos, ext, surf, kind in gs.surface_edits(n, 40, 5):
        box = ref.grid_inject_builtin(g, pos, ext, surf, kind)
        st["inject_surface"].append({"box": [float(v) for v in box], "dense": golden_hash.input_digest(*ref.grid_to_dense(g))})
    ref.grid_destroy(g)
    g = ref.grid_create_builtin(n, capi.Surface.terrain(n))
    st["inject_material"] = []
    for pos, ext, material, add in gs.material_edits(n, 30, 11):
        box = ref.grid_inject_material(g, pos, ext, material, add)
        st["inject_material"].append({"box": [float(v) for v in box], "dense": golden_hash.input_digest(*ref.grid_to_dense(g))})
    ref.grid_destroy(g)
    return out


def main():
    ref = harness.reference()
    for name, make in (("reference_hashes.json", reference_hashes), ("reference_runs.json", reference_runs)):
        out = make(ref)
        with open(os.path.join(HERE, name), "w") as f:
            json.dump(out, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
