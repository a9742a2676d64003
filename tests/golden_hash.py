"""Canonical digests of a LevelDump (see tests/golden/make_golden.py)."""
import hashlib

import numpy as np


def _h(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def input_digest(dist, mat, blend):
    return _h(dist, mat, blend)


def level_digests(lv):
    """exact = everything that must be bit-exact; normals separately (contract tolerance 1e-5, 0 ULP observed)."""
    r = lv.rows
    return {
        "counts": [int(len(r)), int(len(lv.verts)), int(len(lv.idx)), int(len(lv.tverts)), int(len(lv.tidx))],
        "exact": _h(r["id"], r["min"], r["max"], r["nv"], r["ni"], r["tnv"], r["tni"],
                    lv.verts["pos"], lv.verts["sec"], lv.verts["tex"], lv.idx,
                    lv.tverts["pos"], lv.tverts["sec"], lv.tverts["tex"], lv.tidx),
        "normals": _h(lv.verts["nrm"], lv.tverts["nrm"]),
    }


def stored(name):
    """A committed file of tests/golden (JSON) made from the reference's own output by tests/golden/make_golden.py."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)) as f:
        return json.load(f)


def reference_run(name):
    """The reference's Polygonizer::Execute on a named input: {"input_sha256", "stats", "levels": [level_digests]}."""
    grids = stored("reference_hashes.json")["grids"]
    return grids[name] if name in grids else stored("reference_runs.json")["runs"][name]


def run_problems(want, result, levels, stats=True, what=""):
    """Mismatches of `levels` LOD levels of a result (anything with .level(l) and .stats) against a stored reference run:
    every bit-exact field and the normals (0 ULP from the reference, within the 1e-5 contract) by digest, counts by value."""
    problems = []
    for l in range(levels):
        got, w = level_digests(result.level(l)), want["levels"][l]
        if got["counts"] != w["counts"]:
            problems.append("%sL%d: counts (blocks, vertices, indices, transition vertices, transition indices) %s, the reference %s"
                            % (what, l, got["counts"], w["counts"]))
        elif got["exact"] != w["exact"]:
            problems.append("%sL%d: block table, positions, texture bytes or indices differ from the reference's" % (what, l))
        elif got["normals"] != w["normals"]:
            problems.append("%sL%d: normals differ in bits from the reference's" % (what, l))
    if stats and [int(v) for v in result.stats] != want["stats"]:
        problems.append("%sstatistics %s, the reference %s" % (what, [int(v) for v in result.stats], want["stats"]))
    return problems
