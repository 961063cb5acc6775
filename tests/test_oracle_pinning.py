"""Pins the plain-C oracle (oracle/bvh_oracle.c) to the reference:
  (1) the reference's own known answers (SURVEY.md §4 / BASELINE.md §2), via committed golden files
      produced by tests/golden/make_golden.py from the unmodified reference;
  (2) the unmodified reference's outputs on seeded scenes, stored as SHA-256 digests by tests/golden/make_ref_digests.py.
Everything is bit-exact: node arrays, prim ids, hit ids, t, u, v and the per-ray step counters."""
import numpy as np
import pytest

from oracle.pyoracle import ANY_HIT, ROBUST, TIE_LOWEST_ID
from tests.conftest import golden
from tests.helpers import assert_hits_equal, digest, ref_digests

MODES = (("lowest", TIE_LOWEST_ID), ("last", 0), ("any", ANY_HIT | TIE_LOWEST_ID), ("robust", ROBUST | TIE_LOWEST_ID))


def test_kat_simple_example(oracle):
    g = golden("kat_simple_example")
    bb, cc = oracle.tri_bboxes_centers(g["tris"])
    tree = oracle.build(bb, cc, quality="medium")           # High = sweep SAH (+ reinsertion, a no-op on 1 node)
    oracle.set_triangles(tree, g["tris"])
    ids, t, u, v = oracle.trace(tree, g["ray"], flags=0)
    _, _, prim_ids = tree.arrays()
    assert int(np.nonzero(prim_ids == ids[0])[0][0]) == int(g["bvh_order_prim"]) == 1
    assert t[0] == 1.0 and v[0] == 0.5 and u[0] == 0.0 and np.signbit(u[0])      # "distance: 1, u=-0, v=0.5"
    assert_hits_equal((ids, t, u, v), (g["orig_id"], g["t"], g["u"], g["v"]), "simple_example")


def test_kat_serialize_44_bytes(oracle):
    g = golden("kat_serialize")
    tree = oracle.build(g["bboxes"], g["centers"], quality="medium")
    blob = oracle.serialize(tree)
    assert len(blob) == 44
    assert blob.hex() == ("0100000002000000" "000080bf0000803f000080bf0000803f0000803f0000803f" "02000000" "0100000000000000")
    assert blob == g["blob"].tobytes()
    back = oracle.deserialize(blob)
    for a, b in zip(back.arrays(), tree.arrays()):
        assert (a == b).all()


def test_kat_cornell_box(oracle):
    g = golden("kat_cornell")
    from bvh_b200 import scenes
    tris = g["tris"]
    assert tris.shape == (36, 9)
    bb, cc = oracle.tri_bboxes_centers(tris)
    tree = oracle.build(bb, cc, quality="medium")
    assert tree.node_count == int(g["node_count"]) == 37
    oracle.set_triangles(tree, tris)
    rays = scenes.primary_rays(1024, 1024, eye=(0, 1, 2), direction=(0, 0, -1), up=(0, 1, 0))
    ids, _, _, _ = oracle.trace(tree, rays, flags=0)
    hit = ids != 0xFFFFFFFF
    assert int(hit.sum()) == int(g["hit_count"]) == 1027152
    assert (np.packbits(hit) == g["hit_mask"]).all()


@pytest.mark.parametrize("name", ["soup2k_f32", "grid2k_f32", "box12_f32", "soup1k_f64", "soup_incoherent_f32"])
def test_golden_scenes(oracle, name):
    """Oracle traversal of the reference's OWN tree (from the fixture) reproduces the reference's
    outputs, including the visit-order dependent last-visited mode and the step counters."""
    g = golden(name)
    tree = oracle.from_arrays(g["ref_bounds"], g["ref_index"], g["ref_prim_ids"])
    assert oracle.check_invariants(tree, 15) == 0
    assert oracle.serialize(tree) == g["ref_serialized"].tobytes()
    oracle.set_triangles(tree, g["tris"])
    bb, cc = oracle.tri_bboxes_centers(g["tris"])
    assert (bb == g["bboxes"]).all() and (cc == g["centers"]).all()
    for mode, flags in MODES:
        ids, t, u, v, st = oracle.trace(tree, g["rays"], flags=flags, stats=True)
        assert_hits_equal((ids, t, u, v), tuple(g[f"{mode}_{k}"] for k in ("ids", "t", "u", "v")), f"{name}/{mode}")
        assert (st == g[f"{mode}_stats"]).all()
    # tree-free brute force agrees with the canonical closest hit of the ROBUST traversal (the fast
    # slab test is not watertight for rays lying exactly in a box face, e.g. the centre column of
    # grid2k whose direction has x == 0 on the x = 0.5 vertex line: there the result is tree-dependent)
    if g["tris"].shape[0] * g["rays"].shape[0] <= 10_000_000:
        bf = oracle.brute_force(g["tris"], g["rays"])
        assert_hits_equal(bf, tuple(g[f"robust_{k}"] for k in ("ids", "t", "u", "v")), f"{name}/brute-force")


@pytest.mark.parametrize("kind,n,dtype", [("soup", 3000, np.float32), ("grid", 3000, np.float32), ("soup", 1500, np.float64)])
@pytest.mark.parametrize("quality", ["low", "medium"])
def test_builders_match_reference(oracle, kind, n, dtype, quality):
    """The restated BinnedSah / SweepSah builders give the reference's exact node array and prim ids
    (serial DefaultBuilder overload, default_builder.h:49-62)."""
    from bvh_b200 import scenes
    want = ref_digests(f"builders/{kind}-{n}-{np.dtype(dtype).name}/{quality}")
    tris = scenes.make_mesh(kind, n, dtype=dtype)
    bo, co = oracle.tri_bboxes_centers(tris)
    assert digest(bo) == want["bboxes"] and digest(co) == want["centers"]
    to = oracle.build(bo, co, quality=quality)
    for name, a in zip(("bounds", "index", "prim_ids"), to.arrays()):
        assert digest(a) == want[name], f"{kind}/{quality}: {name} differs from the reference's"
    assert oracle.check_invariants(to, 8) == 0
    assert digest(oracle.serialize(to)) == want["serialized"]
    oracle.set_triangles(to, tris)
    rays = scenes.make_primary(kind, 96, 96, dtype=dtype)
    for mode, flags in MODES:
        a = oracle.trace(to, rays, flags=flags, stats=True)
        for name, got in zip(("ids", "t", "u", "v", "stats"), a):
            assert digest(got) == want[f"{mode}_{name}"], f"{kind}/{quality}/{mode}: {name} differs from the reference's"


def test_refit_matches_reference(oracle):
    from bvh_b200 import scenes
    want = ref_digests("refit")
    tris = scenes.soup(2000)
    bb, cc = oracle.tri_bboxes_centers(tris)
    bounds, idx, ids = oracle.build(bb, cc, quality="medium").arrays()        # the reference's tree (pinned above)
    assert digest(bounds) == want["bounds"] and digest(idx) == want["index"] and digest(ids) == want["prim_ids"]
    rng = np.random.RandomState(3)
    leaf = (idx & 15) != 0
    noisy = bounds.copy()
    noisy[leaf] += rng.uniform(-0.01, 0.01, size=noisy[leaf].shape).astype(np.float32)
    noisy[~leaf] = 0
    a = oracle.from_arrays(noisy, idx, ids)
    oracle.refit(a)
    assert digest(a.arrays()[0]) == want["refitted"]


def test_morton_matches_reference(oracle):
    rng = np.random.RandomState(7)
    m32, m64 = [], []
    for _ in range(500):
        x, y, z = (int(v) for v in rng.randint(0, 1 << 10, 3))
        m32.append(oracle.morton_encode(x, y, z, 32))
        x, y, z = (int(v) for v in rng.randint(0, 1 << 21, 3))
        m64.append(oracle.morton_encode(x, y, z, 64))
    want = ref_digests("morton")
    assert digest(np.array(m32, np.uint32)) == want["code32"] and digest(np.array(m64, np.uint64)) == want["code64"]


def test_fma_configuration(oracle):
    # the pinned build flags make fast_mul_add a true FMA (utils.h:75-76); the device code assumes it
    assert oracle.fast_mul_add_is_fma()
