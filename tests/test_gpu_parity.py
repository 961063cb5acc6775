"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C ABI, against the oracle, the
committed golden vectors of the unmodified reference, and — when present — the reference's own example programs.
Bit-exact everywhere: ids, t, u, v (float and double), node arrays, step counters."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from bvh_b200 import scenes
from oracle.pyoracle import ANY_HIT as O_ANY, ROBUST as O_ROBUST, TIE_LOWEST_ID as O_LOWEST
from tests.conftest import golden
from tests.helpers import INVALID, assert_hits_conservative, assert_hits_equal, digest, hits_tuple, ref_digests

pytestmark = pytest.mark.gpu

GOLDEN_SCENES = ["soup2k_f32", "grid2k_f32", "box12_f32", "soup1k_f64", "soup_incoherent_f32"]


def modes(api):
    """(golden key, oracle flags, C-ABI flags)"""
    return (("lowest", O_LOWEST, 0), ("last", 0, api.TIE_LAST_VISITED),
            ("any", O_ANY | O_LOWEST, api.ANY_HIT), ("robust", O_ROBUST | O_LOWEST, api.ROBUST))


@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_lbvh_vs_reference_golden(gpu_lib, name):
    """GPU-built LBVH + GPU traversal reproduce the reference's closest hits on the reference's own
    (different) tree under the canonical tie-break; any-hit agrees on occlusion."""
    api = gpu_lib
    g = golden(name)
    bvh = api.Bvh.build_triangles(g["tris"])
    for kernel in (0,) + api.KERNELS:
        hits = bvh.intersect_rays(g["rays"], flags=kernel)
        assert_hits_equal(hits_tuple(hits), tuple(g[f"lowest_{k}"] for k in ("ids", "t", "u", "v")), f"{name}/closest/{kernel}")
    if g["tris"].dtype == np.float32:
        # the compressed 4-wide path is conservative: where the reference's fast slab test is not watertight
        # (rays lying exactly in a box face; fast and robust golden answers differ) it agrees with robust
        hits = hits_tuple(bvh.intersect_rays(g["rays"], flags=api.KERNEL_WIDE))
        degenerate = g["lowest_ids"] != g["robust_ids"]
        want = tuple(np.where(degenerate, g[f"robust_{k}"], g[f"lowest_{k}"]) for k in ("ids", "t", "u", "v"))
        assert_hits_equal(hits, want, f"{name}/closest/wide")
        occl = bvh.intersect_rays(g["rays"], flags=api.KERNEL_WIDE | api.ANY_HIT)
        assert (((occl["prim_id"] != INVALID) == (g["any_ids"] != INVALID)) | degenerate).all()
    for kernel in (0,) + api.KERNELS:
        hits = bvh.intersect_rays(g["rays"], flags=kernel | api.ROBUST)
        assert_hits_equal(hits_tuple(hits), tuple(g[f"robust_{k}"] for k in ("ids", "t", "u", "v")), f"{name}/robust/{kernel}")
        occl = bvh.intersect_rays(g["rays"], flags=kernel | api.ANY_HIT)
        assert ((occl["prim_id"].astype(np.uint32) != INVALID) == (g["any_ids"] != INVALID)).all()
        miss = occl["prim_id"].astype(np.uint32) == INVALID
        assert (occl["t"][miss] == g["rays"][miss, 7]).all()


@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_reference_tree_on_gpu(gpu_lib, name):
    """The reference's own tree, loaded through bvhNN_load (reference file format) and traced on the
    GPU, gives the reference's outputs in EVERY mode — including the visit-order dependent
    last-visited tie rule and the per-ray step counters: same nodes visited in the same order."""
    api = gpu_lib
    g = golden(name)
    dtype = g["tris"].dtype
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ref.bvh")
        open(path, "wb").write(g["ref_serialized"].tobytes())
        bvh = api.Bvh.load(path, dtype=dtype)
        assert bvh.node_count == g["ref_bounds"].shape[0]
        bounds, index_values, prim_ids = bvh.arrays()
        assert (bounds == g["ref_bounds"]).all() and (index_values == g["ref_index"]).all() and (prim_ids == g["ref_prim_ids"]).all()
        bvh.set_triangles(g["tris"])
        for mode, _, flags in modes(api):
            hits, st = bvh.intersect_rays(g["rays"], flags=flags, stats=True)
            assert_hits_equal(hits_tuple(hits), tuple(g[f"{mode}_{k}"] for k in ("ids", "t", "u", "v")), f"{name}/{mode}")
            want = g[f"{mode}_stats"]
            assert (st["inner_steps"] == want[:, 0]).all() and (st["leaves"] == want[:, 1]).all() and (st["prim_tests"] == want[:, 2]).all()
            for variant in (0,) + api.KERNELS[:3]:                    # persistent kernels, same answers
                hits2 = bvh.intersect_rays(g["rays"], flags=flags | variant)
                assert_hits_equal(hits_tuple(hits2), hits_tuple(hits), f"{name}/{mode}/persistent/{variant}")
        # save -> byte-identical file
        out = os.path.join(tmp, "out.bvh")
        bvh.save(out)
        assert open(out, "rb").read() == g["ref_serialized"].tobytes()


@pytest.mark.parametrize("quality", ["low", "high"])
@pytest.mark.parametrize("kind,n,dtype", [("soup", 20000, np.float32), ("grid", 20000, np.float32), ("soup", 8000, np.float64)])
def test_gpu_tree_is_a_valid_reference_bvh(gpu_lib, oracle, emul, kind, n, dtype, quality):
    """Download the GPU-built tree through the reference accessors: structure invariants hold, boxes are
    what the reference's refit computes, it equals the host emulation's tree node for node, and the
    oracle (reference algorithm) traversing it agrees with the GPU bit for bit, counters included."""
    api = gpu_lib
    tris = scenes.make_mesh(kind, n, dtype=dtype)
    bvh = api.Bvh.build_triangles(tris, quality=quality)
    assert (bvh.get_property("treelets") > 0) == (quality != "low")
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    assert oracle.check_invariants(tree, 8) == 0
    before = tree.arrays()[0]
    oracle.refit(tree)
    assert (tree.arrays()[0] == before).all()
    etree = emul.build(tris=tris, quality=quality)
    eb, ei = emul.compact(etree)
    assert eb.shape == bounds.shape and (eb == bounds).all() and (ei == index_values).all()
    assert (etree["prim_ids"] == prim_ids).all()
    assert bvh.depth == etree["depth"]
    oracle.set_triangles(tree, tris)
    rays = scenes.make_primary(kind, 129, 127, dtype=dtype)
    for mode, oflags, flags in modes(api):
        hits, st = bvh.intersect_rays(rays, flags=flags, stats=True)
        want = oracle.trace(tree, rays, flags=oflags, stats=True)
        assert_hits_equal(hits_tuple(hits), want[:4], f"{kind}/{mode}")
        assert (st["inner_steps"] == want[4][:, 0]).all() and (st["prim_tests"] == want[4][:, 2]).all()
        assert_hits_equal(hits_tuple(bvh.intersect_rays(rays, flags=flags)), want[:4], f"{kind}/{mode}/persistent")
    # bvhNN_refit on an untouched tree changes nothing; the device copy stays usable
    bvh.refit()
    assert (bvh.arrays()[0] == bounds).all()
    assert_hits_equal(hits_tuple(bvh.intersect_rays(rays)), oracle.trace(tree, rays, flags=O_LOWEST)[:4], "after refit")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_wide_morton_keys_match_the_emulation(gpu_lib, emul, monkeypatch, dtype):
    """The 63-bit Morton path (64-bit keys, 8 radix passes; the automatic choice from 2^22 primitives on),
    forced at a size the host emulation handles: same tree node for node."""
    tris = scenes.soup(30000, seed=9).astype(dtype)
    gpu_lib.set_option("morton_bits", 63)
    try:
        bvh = gpu_lib.Bvh.build_triangles(tris)
    finally:
        gpu_lib.set_option("morton_bits", 0)
    assert bvh.get_property("morton_bits") == 63
    bounds, index_values, prim_ids = bvh.arrays()
    etree = emul.build(tris=tris, morton_bits=63, quality="high")
    eb, ei = emul.compact(etree)
    assert eb.shape == bounds.shape and (eb == bounds).all() and (ei == index_values).all()
    assert (etree["prim_ids"] == prim_ids).all()
    narrow = gpu_lib.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 200, 200, dtype=dtype)
    assert_hits_equal(hits_tuple(bvh.intersect_rays(rays)), hits_tuple(narrow.intersect_rays(rays)), "63-bit vs 30-bit tree")


def test_ten_million_triangles_config4(gpu_lib, oracle):
    """BASELINE config 4's mesh size on one GPU: 10M triangles (64-bit Morton keys, 20M node slots), a 4M-ray
    primary batch; structure invariants on the downloaded tree, hit properties, and an exact check of a
    sample against the reference algorithm on the same tree."""
    api = gpu_lib
    n = 10_000_000
    tris = scenes.soup(n)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 2000, 2000)
    hits = bvh.intersect_rays(rays)
    hit = hits["prim_id"] != INVALID
    assert 0.3 < hit.mean() <= 1.0 and (hits["prim_id"][hit] < n).all()
    assert (hits["t"][~hit] == rays[~hit, 7]).all() and (hits["t"][hit] > 0).all()
    bounds, index_values, prim_ids = bvh.arrays()
    assert np.array_equal(np.sort(prim_ids), np.arange(n, dtype=prim_ids.dtype))
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    assert oracle.check_invariants(tree, 8) == 0
    oracle.set_triangles(tree, tris)
    sample = np.sort(np.random.RandomState(4).choice(rays.shape[0], 5000, replace=False))
    want = oracle.trace(tree, rays[sample], flags=O_LOWEST)
    assert_hits_equal(hits_tuple(hits[sample]), want, "soup-10M sample vs oracle")
    wide = bvh.intersect_rays(rays[sample], flags=api.KERNEL_WIDE)
    assert_hits_conservative(wide, want, tris, rays[sample], oracle, "soup-10M sample, wide path vs oracle")


def test_build_from_boxes_and_centres(gpu_lib, oracle):
    """bvh3f_build(pool, bboxes, centers, n, config) — the reference's own entry point — builds the same
    tree as the fused triangle path; bvh3f_set_triangles makes it traceable."""
    api = gpu_lib
    tris = scenes.soup(5000)
    bb, cc = oracle.tri_bboxes_centers(tris)
    a = api.Bvh.build_triangles(tris)
    pool = api.lib().bvh_thread_pool_create(0)
    b = api.Bvh.build(bb, cc, thread_pool=pool)
    api.lib().bvh_thread_pool_destroy(pool)
    for x, y in zip(a.arrays(), b.arrays()):
        assert (x == y).all()
    b.set_triangles(tris)
    rays = scenes.make_primary("soup", 100, 100)
    assert_hits_equal(hits_tuple(a.intersect_rays(rays)), hits_tuple(b.intersect_rays(rays)), "boxes vs triangles")


@pytest.mark.parametrize("n", [1, 2, 3, 5, 33])
def test_tiny_inputs(gpu_lib, oracle, n):
    api = gpu_lib
    tris = scenes.soup(n, seed=n)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 31, 33)
    assert_hits_equal(hits_tuple(bvh.intersect_rays(rays, flags=api.ROBUST)), oracle.brute_force(tris, rays), f"n={n}")
    bounds, index_values, prim_ids = bvh.arrays()
    assert oracle.check_invariants(oracle.from_arrays(bounds, index_values, prim_ids), 8) == 0


@pytest.mark.parametrize("m", [0, 1, 31, 32, 33, 127, 129, 1000])
def test_ragged_ray_counts(gpu_lib, m):
    api = gpu_lib
    g = golden("soup2k_f32")
    bvh = api.Bvh.build_triangles(g["tris"])
    rays = g["rays"][:m]
    hits = bvh.intersect_rays(rays) if m else bvh.intersect_rays(np.zeros((0, 8), np.float32))
    assert hits.shape[0] == m
    assert_hits_equal(hits_tuple(hits), tuple(g[f"lowest_{k}"][:m] for k in ("ids", "t", "u", "v")), f"m={m}")


def test_nan_and_degenerate_rays(gpu_lib, oracle):
    """NaN tmin/tmax (never hit in the reference: every comparison fails), zero directions, inverted and
    empty intervals, infinite tmax — against the oracle traversing the same tree."""
    api = gpu_lib
    tris = scenes.soup(3000)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 40, 40).copy()
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    rays[0::10, 6] = nan
    rays[1::10, 7] = nan
    rays[2::10, 3:6] = 0
    rays[3::10, 6], rays[3::10, 7] = 1.0, 0.5
    rays[4::10, 7] = inf
    rays[5::10, 6] = rays[5::10, 7] = 0.75
    rays[6::10, 3] = 0
    rays[7::10, 3:5] = 0
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    oracle.set_triangles(tree, tris)
    for mode, oflags, flags in modes(api):
        want = oracle.trace(tree, rays, flags=oflags)
        for variant in (0,) + api.KERNELS:
            got = hits_tuple(bvh.intersect_rays(rays, flags=flags | variant))
            nan_rays = np.isnan(rays[:, 7])
            assert (got[0] == want[0]).all()
            ok = ~nan_rays
            assert_hits_equal(tuple(x[ok] for x in got), tuple(x[ok] for x in want), f"{mode}/{variant}")
            assert np.isnan(got[1][nan_rays]).all()           # a miss reports the ray's own tmax


def test_duplicates_degenerates_and_leaf_config(gpu_lib, oracle):
    api = gpu_lib
    base = scenes.soup(1, seed=5)
    tris = np.repeat(base, 300, axis=0)
    tris[100:200, 3:6] = tris[100:200, 0:3]
    tris[100:200, 6:9] = tris[100:200, 0:3]
    more = scenes.soup(2000, seed=9)
    tris = np.concatenate([tris, more])
    rays = scenes.make_primary("soup", 64, 64)
    want = oracle.brute_force(tris, rays)
    for min_leaf, max_leaf in ((None, None), (1, 1), (2, 4), (1, 15)):
        bvh = api.Bvh.build_triangles(tris, min_leaf_size=min_leaf, max_leaf_size=max_leaf)
        assert_hits_equal(hits_tuple(bvh.intersect_rays(rays, flags=api.ROBUST)), want, f"leaf {min_leaf},{max_leaf}")
        bounds, index_values, prim_ids = bvh.arrays()
        assert oracle.check_invariants(oracle.from_arrays(bounds, index_values, prim_ids), max_leaf or 8) == 0


def test_per_ray_callback_api(gpu_lib):
    """bvh3f_intersect_ray with a C leaf callback (reference c_api/bvh.h:233-295) on a GPU-built tree:
    same closest hits as the batched kernel."""
    api = gpu_lib
    g = golden("soup2k_f32")
    tris, rays = g["tris"], g["rays"][:512]
    bvh = api.Bvh.build_triangles(tris)
    _, _, prim_ids = bvh.arrays()
    batched = bvh.intersect_rays(rays)
    state = {}

    def moller(tri, ray, tmax):
        p0, p1, p2 = tri[0:3], tri[3:6], tri[6:9]
        e1, e2 = p0 - p1, p2 - p0
        n = np.cross(e1, e2)
        c = p0 - ray[0:3]
        r = np.cross(ray[3:6], c)
        det = np.dot(n, ray[3:6])
        if det == 0:
            return None
        inv = 1.0 / det
        u, v = np.dot(r, e2) * inv, np.dot(r, e1) * inv
        if u >= -1e-7 and v >= -1e-7 and 1 - u - v >= -1e-7:
            t = np.dot(n, c) * inv
            if ray[6] <= t <= tmax:
                return t
        return None

    CB = C.CFUNCTYPE(C.c_bool, C.c_void_p, C.POINTER(C.c_float), C.c_size_t, C.c_size_t)

    def leaf(_, t_ptr, begin, end):
        was_hit = False
        for i in range(begin, end):
            pid = int(prim_ids[i])
            t = moller(tris[pid].astype(np.float64), state["ray"].astype(np.float64), t_ptr[0])
            if t is not None:
                t_ptr[0] = t
                state["id"] = pid
                was_hit = True
        return was_hit

    class Callback(C.Structure):
        _fields_ = [("user_data", C.c_void_p), ("user_fn", CB)]

    cb = Callback(None, CB(leaf))
    fn = api.lib().bvh3f_intersect_ray
    agree = 0
    for i in range(rays.shape[0]):
        state["ray"], state["id"] = rays[i], INVALID
        fn(bvh.handle, C.c_void_p(rays[i].ctypes.data), C.byref(cb))
        agree += int(state["id"] == int(batched["prim_id"][i]))
    assert agree >= rays.shape[0] - 2        # the python triangle test is float64: allow grazing-edge flips


def test_device_pointers_on_torch_stream(gpu_lib):
    """BVH_DEVICE_POINTERS: rays and hits stay on the device, work is ordered on the caller's stream."""
    import torch
    api = gpu_lib
    g = golden("soup2k_f32")
    api.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        verts = torch.from_numpy(g["tris"]).cuda()
        bvh = api.Bvh.build_triangles(verts.data_ptr(), count=verts.shape[0], dtype=np.float32, flags=api.DEVICE_POINTERS)
        rays = torch.from_numpy(g["rays"]).cuda()
        hits = torch.empty((rays.shape[0], 4), dtype=torch.int32, device="cuda")
        bvh.intersect_rays(rays.data_ptr(), count=rays.shape[0], hits=hits.data_ptr(), flags=api.DEVICE_POINTERS)
        torch.cuda.synchronize()
        out = hits.cpu().numpy().view(api.HIT3F).reshape(-1)
        assert_hits_equal(hits_tuple(out), tuple(g[f"lowest_{k}"] for k in ("ids", "t", "u", "v")), "device pointers")
    finally:
        api.set_stream(None)


@pytest.mark.parametrize("kind", ["soup", "grid"])
def test_full_size_properties(gpu_lib, oracle, kind):
    """BASELINE configs 2/3 at full size (1M triangles, 10M rays): size-independent properties plus an
    exact check of a 20k-ray sample against the reference algorithm on the downloaded tree and against the
    reference's own High-quality tree."""
    api = gpu_lib
    tris = scenes.make_mesh(kind, 1_000_000)
    n = tris.shape[0]
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary(kind, 3163, 3163)
    m = rays.shape[0]
    hits = bvh.intersect_rays(rays)                                 # the library's default path: the exact binary traversal
    assert bvh.properties()["last_kernel"].startswith("trace_persistent_kernel<kTma=")    # exact binary traversal (either ray staging)
    ids = hits["prim_id"]
    hit = ids != INVALID
    assert 0.3 < hit.mean() <= 1.0
    assert (ids[hit] < n).all()
    assert (hits["t"][~hit] == rays[~hit, 7]).all() and (hits["t"][hit] > 0).all()
    assert (hits["u"][hit] >= -1e-6).all() and (hits["v"][hit] >= -1e-6).all() and ((hits["u"] + hits["v"])[hit] <= 1 + 1e-5).all()
    # all binary kernels agree exactly
    for variant in api.KERNELS:
        other = bvh.intersect_rays(rays, flags=variant)
        assert (other.view(np.uint8) == hits.view(np.uint8)).all(), variant
    # the compressed 4-wide path is conservative: every ray / triangle pair the fast binary traversal tests is
    # tested here too, so it may only differ where the fast slab test is not watertight (a hit point exactly on
    # a box face: the leaf holding the other triangle of a shared edge is culled by one ulp), and there it can
    # only report a closer hit, or the same distance with a lower id — and that hit must be a real one
    wide = bvh.intersect_rays(rays, flags=api.KERNEL_WIDE)
    assert bvh.properties()["last_kernel"] == "trace_wide_kernel"
    differs = np.nonzero((wide.view(np.uint8).reshape(m, 16) != hits.view(np.uint8).reshape(m, 16)).any(axis=1))[0]
    assert differs.size < 1e-5 * m, differs.size
    for i in differs:
        w, h = wide[i], hits[i]
        assert w["prim_id"] != INVALID
        assert w["t"] < h["t"] or (w["t"] == h["t"] and w["prim_id"] < h["prim_id"])
        one = oracle.brute_force(tris[w["prim_id"]:w["prim_id"] + 1], rays[i:i + 1])
        assert one[0][0] == 0 and one[1][0] == w["t"] and one[2][0] == w["u"] and one[3][0] == w["v"]
    # nothing lies in front of a reported closest hit: re-trace with tmax just below t as any-hit
    sel = np.nonzero(hit)[0][:: max(1, int(hit.sum()) // 200_000)]
    shortened = rays[sel].copy()
    shortened[:, 7] = hits["t"][sel] * np.float32(1 - 1e-5)
    occl = bvh.intersect_rays(shortened, flags=api.ANY_HIT)
    assert (occl["prim_id"] == INVALID).mean() > 0.999
    # ... and the hit itself is found again as an occluder when tmax is just beyond the reported t
    # (with tmax == t exactly the fast box test may cull the leaf by one ulp: box entry vs triangle t)
    exact = rays[sel].copy()
    exact[:, 7] = hits["t"][sel] * np.float32(1 + 1e-5)
    occl = bvh.intersect_rays(exact, flags=api.ANY_HIT)
    assert (occl["prim_id"] != INVALID).all()
    # exact check of a sample against the oracle on the same tree
    rng = np.random.RandomState(1)
    sample = np.sort(rng.choice(m, 20_000, replace=False))
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    assert oracle.check_invariants(tree, 8) == 0
    oracle.set_triangles(tree, tris)
    want = oracle.trace(tree, rays[sample], flags=O_LOWEST)
    assert_hits_equal(hits_tuple(hits[sample]), want, f"{kind}-1M sample vs oracle")
    assert_hits_conservative(wide[sample], want, tris, rays[sample], oracle, f"{kind}-1M wide path vs oracle")
    # the same sample traced by the unmodified reference on its own High-quality tree (tests/golden/make_ref_digests.py):
    # identical records (the wide path's agreement with the default path is checked above on every ray)
    ref = ref_digests(f"full_size/{kind}")
    for field, a in zip(("ids", "t", "u", "v"), hits_tuple(hits[sample])):
        assert digest(a) == ref[field], f"{kind}-1M sample: {field} differs from the reference's own tree"


def test_incoherent_any_hit_full_size(gpu_lib, oracle):
    """BASELINE config 3: 1M-triangle soup, incoherent AO-style rays, any-hit: occlusion agrees with the
    oracle on a sample; a ray reported occluded really has a hit within [tmin, tmax]."""
    api = gpu_lib
    tris = scenes.soup(1_000_000)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.incoherent_rays(tris, 2_000_000)
    occl = bvh.intersect_rays(rays, flags=api.ANY_HIT | api.KERNEL_TMA)
    closest = bvh.intersect_rays(rays, flags=api.KERNEL_TMA)
    assert ((occl["prim_id"] != INVALID) == (closest["prim_id"] != INVALID)).all()
    wide_occl = bvh.intersect_rays(rays, flags=api.ANY_HIT | api.KERNEL_WIDE)
    wide_closest = bvh.intersect_rays(rays, flags=api.KERNEL_WIDE)
    assert ((wide_occl["prim_id"] != INVALID) == (occl["prim_id"] != INVALID)).all()
    assert (wide_closest.view(np.uint8) == closest.view(np.uint8)).all()
    hit = occl["prim_id"] != INVALID
    assert (occl["t"][hit] <= rays[hit, 7]).all() and (occl["t"][hit] >= closest["t"][hit]).all()
    sample = np.arange(0, rays.shape[0], 100)
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    oracle.set_triangles(tree, tris)
    want = oracle.trace(tree, rays[sample], flags=O_ANY | O_LOWEST)
    assert_hits_equal(hits_tuple(occl[sample]), want, "incoherent any-hit sample")


def test_double_precision_config5(gpu_lib, oracle):
    """BASELINE config 5: Node<double,3>, 100K triangles, 1M rays, exact against the oracle."""
    api = gpu_lib
    tris = scenes.soup(100_000, dtype=np.float64)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 1000, 1000, dtype=np.float64)
    hits = bvh.intersect_rays(rays)
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    assert oracle.check_invariants(tree, 8) == 0
    oracle.set_triangles(tree, tris)
    sample = np.arange(0, rays.shape[0], 25)
    want = oracle.trace(tree, rays[sample], flags=O_LOWEST)
    assert_hits_equal(hits_tuple(hits[sample]), want, "double")
    simple = bvh.intersect_rays(rays, flags=api.KERNEL_SIMPLE)
    assert (simple.view(np.uint8) == hits.view(np.uint8)).all()


def test_reference_c_example_runs_unmodified(gpu_lib, tmp_path):
    """The reference's own test/c_api_example.c (+ load_obj.cpp), compiled UNMODIFIED against this
    repository's <bvh/v2/c_api/bvh.h> and linked to libbvh_c.so (oracle/Makefile target c_api_example, built
    into oracle/_ref/ where the reference's sources exist; skipped elsewhere).  It builds with bvh3f_build on the GPU
    and traces 1024x1024 rays through bvh3f_intersect_ray + its C leaf callback: the reference's ctest
    known answer is 1 027 152 intersections (SURVEY.md §4)."""
    import re
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "c_api_example")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/c_api_example was not built (needs the reference's sources at build time)")
    tris = golden("kat_cornell")["tris"]
    obj = tmp_path / "cornell.obj"
    with open(obj, "w") as f:
        for t in tris:
            for k in range(3):
                f.write("v %.9g %.9g %.9g\n" % tuple(t[3 * k:3 * k + 3]))
        for i in range(tris.shape[0]):
            f.write("f %d %d %d\n" % (3 * i + 1, 3 * i + 2, 3 * i + 3))
    out = subprocess.run([exe, str(obj), "--eye", "0", "1", "2", "--dir", "0", "0", "-1", "--up", "0", "1", "0",
                          "-o", str(tmp_path / "render.ppm")], capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stderr
    m = re.search(r"(\d+) intersection\(s\) found", out.stdout)
    assert m and int(m.group(1)) == 1027152, out.stdout


def _write_cornell_obj(path):
    tris = golden("kat_cornell")["tris"]
    with open(path, "w") as f:
        for t in tris:
            for k in range(3):
                f.write("v %.9g %.9g %.9g\n" % tuple(t[3 * k:3 * k + 3]))
        for i in range(tris.shape[0]):
            f.write("f %d %d %d\n" % (3 * i + 1, 3 * i + 2, 3 * i + 3))


def test_reference_cxx_examples_run_unmodified(gpu_lib, tmp_path):
    """The reference's own C++ test programs — test/simple_example.cpp, test/serialize.cpp and
    test/benchmark.cpp (+ load_obj.cpp) — compiled UNMODIFIED against this repository's <bvh/v2/*.h> surface
    (oracle/Makefile target cxx_examples, built into oracle/_ref/ where the reference's sources exist).  DefaultBuilder::build runs on
    the GPU; the ctest pass criteria of the reference (exit code 0) and its known answers must hold:
    simple_example hits at distance 1 with v = 0.5; serialize round-trips; the Cornell-box benchmark finds
    1 027 152 intersections (SURVEY.md §4)."""
    import re
    import subprocess
    build_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")
    exes = {n: os.path.join(build_dir, "cxx_" + n) for n in ("simple_example", "serialize", "benchmark")}
    if not all(os.path.exists(e) for e in exes.values()):
        pytest.skip("oracle/_ref/cxx_* were not built (needs the reference's sources at build time)")
    out = subprocess.run([exes["simple_example"]], capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "Intersection found" in out.stdout and re.search(r"distance: 1\b", out.stdout) and "0.5" in out.stdout, out.stdout
    out = subprocess.run([exes["serialize"]], capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert out.returncode == 0 and "same as the original" in out.stdout, out.stdout + out.stderr
    obj = tmp_path / "cornell.obj"
    _write_cornell_obj(obj)
    out = subprocess.run([exes["benchmark"], str(obj), "--eye", "0", "1", "2", "--dir", "0", "0", "-1", "--up", "0", "1", "0"],
                         capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stdout + out.stderr
    m = re.search(r"(\d+) intersection\(s\) found", out.stdout)
    assert m and int(m.group(1)) == 1027152, out.stdout
    assert re.search(r"Built BVH with \d+ node\(s\)", out.stdout)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gpu_refit_after_vertices_move(gpu_lib, oracle, dtype):
    """bvhNN_refit_triangles: after moving the vertices the GPU recomputes leaf and inner boxes exactly as
    the reference's refit does from the new leaf boxes (same topology, bit-identical bounds), and tracing
    the refitted tree gives the brute-force answer for the moved mesh."""
    api = gpu_lib
    tris = scenes.soup(6000, dtype=dtype)
    bvh = api.Bvh.build_triangles(tris)
    _, index_before, ids_before = bvh.arrays()
    rng = np.random.RandomState(4)
    moved = (tris.reshape(-1, 3, 3) + rng.uniform(-0.02, 0.02, size=(tris.shape[0], 1, 3))).reshape(-1, 9).astype(dtype)
    bvh.refit_triangles(moved)
    bounds, index_values, prim_ids = bvh.arrays()
    assert (index_values == index_before).all() and (prim_ids == ids_before).all()
    # expected: leaf boxes from the moved triangles (in leaf order), inner boxes by the reference's refit
    want = bounds.copy()
    bb, _ = oracle.tri_bboxes_centers(moved)
    for i in np.nonzero((index_values & 15) != 0)[0]:
        first, count = int(index_values[i]) >> 4, int(index_values[i]) & 15
        boxes = bb[prim_ids[first:first + count].astype(np.int64)]
        want[i, 0::2] = boxes[:, 0:3].min(axis=0)
        want[i, 1::2] = boxes[:, 3:6].max(axis=0)
    want[(index_values & 15) == 0] = 0
    tree = oracle.from_arrays(want, index_values, prim_ids)
    oracle.refit(tree)
    assert (tree.arrays()[0] == bounds).all()
    rays = scenes.make_primary("soup", 80, 80, dtype=dtype)
    assert_hits_equal(hits_tuple(bvh.intersect_rays(rays, flags=api.ROBUST)), oracle.brute_force(moved, rays), "refit trace")


@pytest.mark.parametrize("dtype,flags_name", [(np.float32, None), (np.float32, "ANY_HIT"), (np.float64, None),
                                              (np.float32, "KERNEL_WIDE"), (np.float32, "KERNEL_NO_TMA"), (np.float32, "KERNEL_TMA")])
def test_gather_entry_point_on_one_gpu(gpu_lib, dtype, flags_name):
    """bvhNN_intersect_rays_gather with both "ranks" on one device: the shard's records must land, identical to
    the plain batched call, in the shard's slot of every gathered array (and nowhere else), and in the local
    array when one is given."""
    import torch
    api = gpu_lib
    tris = scenes.soup(20000, seed=2).astype(dtype)
    bvh = api.Bvh.build_triangles(tris)
    rays = scenes.make_primary("soup", 301, 211, dtype=dtype)          # 63 511 rays: a ragged last chunk
    if flags_name in ("KERNEL_WIDE", "KERNEL_TMA"):                    # incoherent order: stragglers hold staging slots (evictions)
        rays = np.ascontiguousarray(rays[np.random.default_rng(5).permutation(rays.shape[0])])
    rays[5, 6] = np.nan                                                # a ray retired in the refill path
    rays[40, 7] = np.nan
    flags = getattr(api, flags_name) if flags_name else 0
    want = bvh.intersect_rays(rays, flags=flags)
    m = rays.shape[0]
    words = want.dtype.itemsize // 4
    d_rays = torch.from_numpy(rays).cuda()
    offset = 1000                                                      # the shard's position in the gathered arrays
    total = m + 2 * offset
    gathered = [torch.full((total, words), 0x5A5A5A5A, dtype=torch.int32, device="cuda") for _ in range(2)]
    expect = np.frombuffer(want.tobytes(), np.int32).reshape(m, words)
    for with_local in (True, False):
        for g in gathered: g.fill_(0x5A5A5A5A)
        local = torch.zeros((m, words), dtype=torch.int32, device="cuda") if with_local else None
        bvh.intersect_rays_gather(d_rays.data_ptr(), m, [g.data_ptr() for g in gathered], offset,
                                  hits_ptr=local.data_ptr() if with_local else 0, flags=flags)
        bvh.sync()
        torch.cuda.synchronize()
        for g in gathered:
            got = g.cpu().numpy()
            assert (got[offset:offset + m] == expect).all()
            assert (got[:offset] == 0x5A5A5A5A).all() and (got[offset + m:] == 0x5A5A5A5A).all()
        if with_local:
            assert (local.cpu().numpy() == expect).all()


@pytest.mark.parametrize("kind,n,dtype", [("soup", 20000, np.float32), ("grid", 20000, np.float32), ("soup", 6000, np.float64),
                                           ("soup", 200, np.float32), ("soup", 64, np.float32), ("soup", 3, np.float32)])
def test_sah_treelets_match_the_emulation(gpu_lib, emul, kind, n, dtype):
    """Quality Medium / High = LBVH + SAH treelet pass: the device runs the same phase code as the host
    emulation, so the compacted trees must be identical, Medium and High build the same tree, and the traversal
    results equal the plain LBVH's (Quality Low)."""
    api = gpu_lib
    tris = (scenes.soup(n, seed=7) if kind == "soup" else scenes.make_mesh(kind, n)).astype(dtype)
    rays = scenes.make_primary(kind, 128, 128, dtype=dtype)
    plain = api.Bvh.build_triangles(tris, quality="low")
    assert plain.get_property("treelets") == 0
    bvh = api.Bvh.build_triangles(tris)                      # library default: Quality High
    medium = api.Bvh.build_triangles(tris, quality="medium")
    assert bvh.get_property("treelets") > 0 and bvh.get_property("quality") == 2
    bounds, index_values, prim_ids = bvh.arrays()
    for x, y in zip(medium.arrays(), (bounds, index_values, prim_ids)):
        assert (x == y).all()
    etree = emul.build(tris=tris, quality="high")
    assert emul.lib.emul_last_treelet_count() == bvh.get_property("treelets")
    eb, ei = emul.compact(etree)
    assert eb.shape == bounds.shape and (eb == bounds).all() and (ei == index_values).all()
    assert (etree["prim_ids"] == prim_ids).all() and bvh.depth == etree["depth"]
    for flags in (api.KERNEL_TMA, api.KERNEL_WIDE, api.KERNEL_SIMPLE):
        assert_hits_equal(hits_tuple(bvh.intersect_rays(rays, flags=flags)), hits_tuple(plain.intersect_rays(rays, flags=flags)),
                          f"treelets vs plain LBVH ({flags})")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,dtype,bits", [("soup", 300_000, np.float32, 30), ("grid", 50_000, np.float32, 63), ("soup", 2049, np.float64, 30)])
def test_build_switches_give_the_same_tree(gpu_lib, kind, n, dtype, bits):
    """The one-sweep radix sort (one kernel per pass, decoupled look-back) and the three-kernel passes must order the
    primitives identically, and the hierarchy kernel's block-local phase must not change the tree: node arrays and
    primitive order equal for every combination of the build switches."""
    api = gpu_lib
    tris = scenes.make_mesh(kind, n, dtype=dtype)
    api.set_option("morton_bits", bits)
    try:
        trees = []
        for onesweep, hierarchy in ((1, 128), (0, 128), (1, 0), (1, 64)):
            api.set_option("sort_onesweep", onesweep)
            api.set_option("hierarchy", hierarchy)
            for _ in range(2):                                   # twice: the look-back must not depend on timing
                bvh = api.Bvh.build_triangles(tris)
                b, ix, ids = bvh.arrays()
                trees.append((b.tobytes(), ix.tobytes(), ids.tobytes()))
        assert all(t == trees[0] for t in trees[1:])
    finally:
        api.set_option("morton_bits", 0)
        api.set_option("sort_onesweep", 1)
        api.set_option("hierarchy", 128)


@pytest.mark.gpu
def test_optimize_on_a_gpu_built_tree(gpu_lib, oracle):
    """bvh3f_optimize on a GPU-built tree (reference ReinsertionOptimizer on the host mirror, re-uploaded before the
    next batched call): the SAH cost of the tree goes down, the invariants hold, batched results do not change."""
    import ctypes as C
    api = gpu_lib
    tris = scenes.soup(60_000, seed=9)
    rays = scenes.make_primary("soup", 300, 300)
    bvh = api.Bvh.build_triangles(tris, quality="low")

    def sah(bounds, index_values):
        d = bounds[:, 1::2].astype(np.float64) - bounds[:, 0::2]
        area = (d[:, 0] + d[:, 1]) * d[:, 2] + d[:, 0] * d[:, 1]
        count = (index_values & 15).astype(np.float64)
        return float(np.where(count > 0, area * count, area).sum() / area[0])

    before_hits = bvh.intersect_rays(rays)
    b0, i0, ids0 = bvh.arrays()
    L = api.lib()
    pool = L.bvh_thread_pool_create(0)
    L.bvh3f_optimize(C.c_void_p(pool), bvh.handle)
    L.bvh_thread_pool_destroy(C.c_void_p(pool))
    b1, i1, ids1 = bvh.arrays()
    assert sah(b1, i1) < sah(b0, i0) and np.array_equal(ids0, ids1) and b1.shape == b0.shape
    tree = oracle.from_arrays(b1, i1, ids1)
    assert oracle.check_invariants(tree, 8) == 0
    after_hits = bvh.intersect_rays(rays)                       # re-uploads the edited mirror
    assert np.array_equal(after_hits, before_hits)
    st_before = api.Bvh.build_triangles(tris, quality="low").intersect_rays(rays, stats=True)[1]
    st_after = bvh.intersect_rays(rays, stats=True)[1]
    # The reference's pass (pinned node for node in tests/test_optimize.py) lowers the SAH cost; on a uniform soup it moves a
    # handful of nodes only (the unmodified reference does exactly the same on this tree), so the step count of a particular
    # camera may go either way by a few steps: it must stay within 1 %.
    assert abs(float(st_after["inner_steps"].sum()) / float(st_before["inner_steps"].sum()) - 1.0) < 0.01


@pytest.mark.gpu
def test_identical_triangles_with_wide_keys(gpu_lib, oracle):
    """10^5 copies of one triangle plus a few others, 63-bit keys: every key of the run is equal, the index tie-break
    must balance the run (depth ~ log2 n, far from the 127 levels the build pass can track), the per-ray entry points
    (whose stack grows beyond the reference's 64 entries when needed) and the batched ones agree with brute force."""
    api = gpu_lib
    base = scenes.soup(8, seed=3)
    tris = np.concatenate([np.repeat(base[:1], 100_000, axis=0), base[1:]]).astype(np.float32)
    api.set_option("morton_bits", 63)
    try:
        bvh = api.Bvh.build_triangles(tris, quality="low")
        assert bvh.get_property("morton_bits") == 63 and bvh.depth < 40
        rays = scenes.make_primary("soup", 24, 24)
        hits = bvh.intersect_rays(rays)
        bf = oracle.brute_force(tris, rays)
        assert_hits_equal(hits_tuple(hits), bf, "identical triangles")
        assert (hits["prim_id"][hits["prim_id"] < 100_000] == 0).all()      # lowest id among the identical ones
        b, ix, ids = bvh.arrays()
        tree = oracle.from_arrays(b, ix, ids)
        assert oracle.check_invariants(tree, 8) == 0
    finally:
        api.set_option("morton_bits", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["soup", "grid"])
def test_wide_kernel_budgets_keep_the_answers(gpu_lib, oracle, kind):
    """The opt-in wide kernel at every round budget, on an incoherent ray order: the binary kernel's closest hits
    except where the binary traversal itself misses a true hit (conservative boxes: the wide path may only find a
    closer real hit, or the same distance with a lower id), the same occluded / not occluded verdict for any-hit, and
    the same answers whatever the budget."""
    api = gpu_lib
    tris = scenes.make_mesh(kind, 150_000)
    rays = scenes.make_primary(kind, 500, 400)
    shuffled = np.ascontiguousarray(rays[np.random.default_rng(3).permutation(rays.shape[0])])
    bvh = api.Bvh.build_triangles(tris)
    want = bvh.intersect_rays(shuffled)
    want_any = bvh.intersect_rays(shuffled, flags=api.ANY_HIT)
    try:
        first = None
        for budget in (1, 4, 0):
            api.set_option("wide_budget", budget)
            got = bvh.intersect_rays(shuffled, flags=api.KERNEL_WIDE)
            assert bvh.properties()["last_kernel"] == "trace_wide_kernel"
            assert_hits_conservative(got, hits_tuple(want), tris, shuffled, oracle, f"wide kernel, budget {budget}", max_fraction=1e-4)
            first = got if first is None else first
            assert np.array_equal(got, first), budget
            got_any = bvh.intersect_rays(shuffled, flags=api.KERNEL_WIDE | api.ANY_HIT)
            assert ((got_any["prim_id"] == INVALID) == (want_any["prim_id"] == INVALID)).mean() > 1 - 1e-4
    finally:
        api.set_option("wide_budget", 4)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sorted_ray_order_keeps_the_answers(gpu_lib, dtype):
    """BVH_SORT_RAYS traverses an incoherent batch in the Morton order of its origins; hits[i] must still answer
    rays[i], bit for bit (closest hit, both kernels) and verdict for verdict (any-hit), NaN origins included."""
    api = gpu_lib
    tris = scenes.soup(100_000, seed=4).astype(dtype)
    rays = scenes.incoherent_rays(tris.astype(np.float32), 200_003, seed=8).astype(dtype)
    rays[17, 0] = np.nan
    bvh = api.Bvh.build_triangles(tris)
    base = bvh.intersect_rays(rays)
    got = bvh.intersect_rays(rays, flags=api.SORT_RAYS)
    assert np.array_equal(got.view(np.uint8), base.view(np.uint8))
    occluded = bvh.intersect_rays(rays, flags=api.ANY_HIT)["prim_id"] != (INVALID if dtype == np.float32 else 0xFFFFFFFFFFFFFFFF)
    got_any = bvh.intersect_rays(rays, flags=api.ANY_HIT | api.SORT_RAYS)["prim_id"] != (INVALID if dtype == np.float32 else 0xFFFFFFFFFFFFFFFF)
    assert np.array_equal(got_any, occluded)
    if dtype == np.float32:
        wide = bvh.intersect_rays(rays, flags=api.KERNEL_WIDE)
        wide_sorted = bvh.intersect_rays(rays, flags=api.KERNEL_WIDE | api.SORT_RAYS)
        assert np.array_equal(wide_sorted.view(np.uint8), wide.view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_traversal_switches_keep_the_answers(gpu_lib, oracle, dtype):
    """Scheduling switches of the persistent kernel — refill threshold, inner budget, size of a warp's private run, ray
    staging (streaming / TMA), stack rounding, shared-memory carve-out — decide WHEN a ray is traversed, never how: the
    hit records (closest hit and any-hit, same tree) must be bit-identical for every setting, and equal to the oracle's."""
    api = gpu_lib
    tris = scenes.soup(120_000, seed=11).astype(dtype)
    rays = np.concatenate([scenes.make_primary("soup", 400, 300), scenes.incoherent_rays(tris.astype(np.float32), 80_003, seed=5)]).astype(dtype)
    bvh = api.Bvh.build_triangles(tris)
    defaults = {"refill_min": 8, "inner_budget": 8, "chunk_rays": 64, "variant": 0, "stack_round": 2, "smem_carveout": -1}
    base = bvh.intersect_rays(rays)
    base_any = bvh.intersect_rays(rays, flags=api.ANY_HIT)
    bounds, index_values, prim_ids = bvh.arrays()
    tree = oracle.from_arrays(bounds, index_values, prim_ids)
    oracle.set_triangles(tree, tris)
    sample = np.arange(0, rays.shape[0], 7)
    assert_hits_equal(hits_tuple(base[sample]), oracle.trace(tree, rays[sample], flags=O_LOWEST), "default switches vs oracle")
    settings = [{"refill_min": 1}, {"refill_min": 32}, {"refill_min": 20, "inner_budget": 1}, {"inner_budget": 0}, {"chunk_rays": 32},
                {"chunk_rays": 1024}, {"variant": 1}, {"variant": 1, "chunk_rays": 256, "refill_min": 3}, {"stack_round": 8},
                {"smem_carveout": 100}, {"smem_carveout": 0}]
    try:
        for setting in settings:
            for name, value in {**defaults, **setting}.items():
                api.set_option(name, value)
            got = bvh.intersect_rays(rays)
            assert np.array_equal(got.view(np.uint8), base.view(np.uint8)), setting
            got_any = bvh.intersect_rays(rays, flags=api.ANY_HIT)
            assert np.array_equal(got_any.view(np.uint8), base_any.view(np.uint8)), setting
    finally:
        for name, value in defaults.items():
            api.set_option(name, value)
