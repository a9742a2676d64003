"""CPU tests of the test infrastructure itself (no GPU): the CPU restatement (oracle/restate) is pinned against the
committed digests of the reference's output (tests/golden, made by tests/golden/make_golden.py); the reference's own
properties are checked against the unmodified reference compiled under oracle/_ref, when that build is present."""
import json
import os

import numpy as np
import pytest

import golden_hash
import grids

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_hashes.json")


def golden():
    with open(GOLDEN) as f:
        return json.load(f)["grids"]


class _Restated:
    """A restatement run seen as a result: .level(l) and .stats."""

    def __init__(self, restatement, h):
        self.level = lambda l: restatement.level(h, l)
        self.stats = restatement.stats(h)


@pytest.mark.parametrize("name", sorted(grids.SMALL))
def test_restatement_matches_reference(restatement, name):
    dist, mat, blend = grids.SMALL[name]()
    want = golden_hash.reference_run(name)
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"]
    h = restatement.run(dist, mat, blend)
    flags = golden_hash.stored("reference_runs.json")["empty_flags"][name]
    assert golden_hash._h(restatement.empty_flags(h, dist.shape[0])) == flags, "BF_Empty rule"
    assert restatement.levels(h) == len(want["levels"])
    problems = golden_hash.run_problems(want, _Restated(restatement, h), len(want["levels"]))   # normals: 0 ULP
    restatement.destroy(h)
    assert not problems, "\n".join(problems)


@pytest.mark.parametrize("name", sorted(grids.SMALL) + ["hostile128"])
def test_restatement_matches_golden_digests(restatement, name):
    dist, mat, blend = (grids.SMALL.get(name) or grids.MEDIUM[name])()
    want = golden()[name]
    assert golden_hash.input_digest(dist, mat, blend) == want["input_sha256"], "test grid generator changed: regenerate the golden file"
    h = restatement.run(dist, mat, blend)
    assert [int(v) for v in restatement.stats(h)] == want["stats"]
    assert restatement.levels(h) == len(want["levels"])
    for l, w in enumerate(want["levels"]):
        got = golden_hash.level_digests(restatement.level(h, l))
        assert got["counts"] == w["counts"], "level %d counts" % l
        assert got["exact"] == w["exact"], "level %d bit-exact fields" % l
        assert got["normals"] == w["normals"], "level %d normals (0 ULP expected on x86-64 without FMA)" % l
    restatement.destroy(h)


def test_reference_determinism_across_threads(reference):
    """The reference is bit-deterministic across OpenMP thread counts (SURVEY.md section 4.3)."""
    dist, mat, blend = grids.SMALL["hostile64"]()
    g = reference.grid_from_dense(dist, mat, blend)
    dumps = []
    for threads in (1, 4):
        s, _ = reference.polygonize(g, threads=threads)
        dumps.append([golden_hash.level_digests(reference.surface_level(s, l)) for l in range(reference.surface_levels(s))])
        reference.surface_destroy(s)
    reference.grid_destroy(g)
    assert dumps[0] == dumps[1]


def test_reference_config1_anchors(reference):
    """BASELINE config 1 (64^3 sphere) through Grid::Create + Polygonizer::Execute: the survey's expected counts."""
    g = reference.grid_sphere(64, (32, 32, 32), 19.2)
    s, _ = reference.polygonize(g, threads=2)
    st = reference.surface_stats(s)
    assert reference.surface_levels(s) == 3 and st[0] == 73 and st[2] == 9096
    l0 = reference.surface_level(s, 0)
    assert len(l0.verts) == 8832 and len(l0.idx) == 41496
    assert int((l0.verts["tex"][:, 0] != 0).sum()) == 0  # Reserved byte is value-initialised to 0
    reference.surface_destroy(s); reference.grid_destroy(g)


def test_terrain_generator_is_deterministic_and_parity_on_it(restatement):
    from voxels_b200 import synth
    d1, m1, b1 = (t.numpy() for t in synth.terrain(64))
    d2, m2, b2 = (t.numpy() for t in synth.terrain(64))
    assert np.array_equal(d1, d2) and np.array_equal(m1, m2) and np.array_equal(b1, b2)
    assert d1.min() == -4 and d1.max() == 4 and set(np.unique(m1)) <= {0, 1, 2, 3}
    want = golden_hash.reference_run("terrain64")
    assert golden_hash.input_digest(d1, m1, b1) == want["input_sha256"]
    h = restatement.run(d1, m1, b1)
    problems = golden_hash.run_problems(want, _Restated(restatement, h), len(want["levels"]), stats=False)
    restatement.destroy(h)
    assert not problems, "\n".join(problems)
