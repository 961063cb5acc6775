"""Runs the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref REF=<reference checkout>`) on the inputs of
the tests that compare with it, and stores what they compare against:

    python tests/golden/make_ref_digests.py

  ref_digests.json   SHA-256 digests (tests/helpers.py digest) of every array a test compares bit for bit, by test case
  ref_topology.npz   what a test needs as INPUT from the reference: the topology (node index words, prim ids) of the trees
                     the reference's C library builds for the 2-D and optimizer tests (tests/helpers.py tree_blob rebuilds
                     the exact file from it), and the reference's per-ray answers of the 2-D callback traversal

Inputs are the tests' own seeded scenes, so the tests rebuild them bit for bit.
"""
import ctypes as C
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from bvh_b200 import scenes  # noqa: E402
from oracle.pyoracle import TIE_LOWEST_ID, Ref  # noqa: E402
from tests import test_c_abi_2d as t2d, test_optimize as topt  # noqa: E402
from tests.helpers import digest, tree_blob  # noqa: E402
from tests.test_oracle_pinning import MODES  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
REF_C = os.path.join(ROOT, "oracle", "_ref", "libbvh_c_ref.so")   # the reference's own C library
ref = Ref()
digests, arrays = {}, {}


class Config(C.Structure):
    """struct bvh_build_config of the reference's C API"""
    _fields_ = [("quality", C.c_int), ("min_leaf_size", C.c_size_t), ("max_leaf_size", C.c_size_t), ("parallel_threshold", C.c_size_t)]


def pinning():
    for kind, n, dtype in (("soup", 3000, np.float32), ("grid", 3000, np.float32), ("soup", 1500, np.float64)):
        for quality in ("low", "medium"):
            tris = scenes.make_mesh(kind, n, dtype=dtype)
            bb, cc = ref.tri_bboxes_centers(tris)
            tree = ref.build(bb, cc, quality=quality, threads=-1)
            bounds, index, ids = tree.arrays()
            d = dict(bboxes=digest(bb), centers=digest(cc), bounds=digest(bounds), index=digest(index), prim_ids=digest(ids),
                     serialized=digest(ref.serialize(tree)))
            ref.set_triangles(tree, tris)
            rays = scenes.make_primary(kind, 96, 96, dtype=dtype)
            for mode, flags in MODES:
                for name, a in zip(("ids", "t", "u", "v", "stats"), ref.trace(tree, rays, flags=flags, stats=True)):
                    d[f"{mode}_{name}"] = digest(a)
            digests[f"builders/{kind}-{n}-{np.dtype(dtype).name}/{quality}"] = d

    tris = scenes.soup(2000)
    bb, cc = ref.tri_bboxes_centers(tris)
    bounds, idx, ids = ref.build(bb, cc, quality="medium", threads=-1).arrays()
    rng = np.random.RandomState(3)
    leaf = (idx & 15) != 0
    noisy = bounds.copy()
    noisy[leaf] += rng.uniform(-0.01, 0.01, size=noisy[leaf].shape).astype(np.float32)
    noisy[~leaf] = 0
    b = ref.from_arrays(noisy, idx, ids)
    ref.refit(b)
    digests["refit"] = dict(bounds=digest(bounds), index=digest(idx), prim_ids=digest(ids), refitted=digest(b.arrays()[0]))

    rng = np.random.RandomState(7)
    m32, m64 = [], []
    for _ in range(500):
        m32.append(ref.morton_encode(*(int(v) for v in rng.randint(0, 1 << 10, 3)), 32))
        m64.append(ref.morton_encode(*(int(v) for v in rng.randint(0, 1 << 21, 3)), 64))
    digests["morton"] = dict(code32=digest(np.array(m32, np.uint32)), code64=digest(np.array(m64, np.uint64)))


def c_abi_2d(tmp):
    for s in ("2f", "2d"):
        api = t2d.Api2(REF_C, s)
        boxes, centers, rays = t2d.scene2(700, 3, api.dtype)
        bvh = api.build(boxes, centers)
        path = os.path.join(tmp, "tree.bin")
        api.save(bvh, path)
        blob = open(path, "rb").read()
        nodes, ids = topt.parse(blob, 2, api.dtype)
        assert tree_blob(nodes["index"], ids, boxes, 2) == blob
        arrays[f"c_abi_2d/{s}/index"], arrays[f"c_abi_2d/{s}/prim_ids"] = nodes["index"], ids
        d = dict(blob=digest(blob), nodes=digest(np.array(api.nodes(bvh), np.float64)))
        prim_ids = api.prim_ids(bvh)
        for variant in ("intersect_ray", "intersect_ray_any", "intersect_ray_robust", "intersect_ray_any_robust"):
            res = api.trace(bvh, rays, boxes, prim_ids, variant)
            arrays[f"c_abi_2d/{s}/{variant}/id"] = np.array([r[0] for r in res], np.int64)
            arrays[f"c_abi_2d/{s}/{variant}/t"] = np.array([np.nan if r[1] is None else r[1] for r in res], np.float64)
            arrays[f"c_abi_2d/{s}/{variant}/calls"] = np.array([r[2] for r in res], np.int64)
        for i in range(api.f("get_node_count")(bvh)):          # the test's leaf-box edit, then the reference's refit
            nd = api.f("get_node")(bvh, i)
            if api.g("is_leaf")(nd):
                b = api.g("get_bbox")(nd)
                b.max.x += 0.25; b.min.y -= 0.125
                api.g("set_bbox")(nd, C.byref(b))
        api.f("refit")(bvh)
        d["refit_nodes"] = digest(np.array(api.nodes(bvh), np.float64))
        api.save(bvh, path)
        d["refit_blob"] = digest(open(path, "rb").read())
        api.f("destroy")(bvh)
        digests[f"c_abi_2d/{s}"] = d


def optimize(tmp):
    lib = C.CDLL(REF_C)
    for s, dim, dtype in (("3f", 3, np.float32), ("3d", 3, np.float64), ("2f", 2, np.float32), ("2d", 2, np.float64)):
        for n in (300, 3000):
            rf = topt.bind(lib, s)
            boxes, centers = topt.scene(dim, n, dtype, 7 + n)
            cfg = Config(1, 1, 8, 1024)                  # Quality::Medium: SweepSAH without the optimizer
            tree = rf("build")(None, boxes.ctypes.data, centers.ctypes.data, n, C.byref(cfg))
            before = topt.save_bytes(rf, tree, os.path.join(tmp, "before.bin"))
            pool = lib.bvh_thread_pool_create(4)
            rf("optimize")(pool if n > 100 else None, tree)
            lib.bvh_thread_pool_destroy(pool)
            after = topt.save_bytes(rf, tree, os.path.join(tmp, "after.bin"))
            rf("destroy")(tree)
            nodes, ids = topt.parse(before, dim, dtype)
            assert tree_blob(nodes["index"], ids, boxes, dim) == before
            want, want_ids = topt.parse(after, dim, dtype)
            arrays[f"optimize/{s}/{n}/index"], arrays[f"optimize/{s}/{n}/prim_ids"] = nodes["index"], ids
            digests[f"optimize/{s}/{n}"] = dict(before=digest(before), after=digest(after), after_nodes=digest(want),
                                                after_prim_ids=digest(want_ids))


def full_size():
    """tests/test_gpu_parity.py test_full_size_properties: the reference's own High-quality tree of the 1M-triangle mesh,
    traced at the test's 20k-ray sample of the 3163 x 3163 camera."""
    for kind in ("soup", "grid"):
        tris = scenes.make_mesh(kind, 1_000_000)
        rays = scenes.make_primary(kind, 3163, 3163)
        sample = np.sort(np.random.RandomState(1).choice(rays.shape[0], 20_000, replace=False))
        bb, cc = ref.tri_bboxes_centers(tris)
        tree = ref.build(bb, cc, quality="high", threads=0)
        ref.set_triangles(tree, tris)
        want = ref.trace(tree, rays[sample], flags=TIE_LOWEST_ID, threads=0)
        digests[f"full_size/{kind}"] = {k: digest(a) for k, a in zip(("ids", "t", "u", "v"), want)}
        print(kind, "sample hits", int((want[0] != 0xFFFFFFFF).sum()), flush=True)


if __name__ == "__main__":
    pinning()
    with tempfile.TemporaryDirectory() as tmp:
        c_abi_2d(tmp)
        optimize(tmp)
    full_size()
    with open(os.path.join(OUT, "ref_digests.json"), "w") as f:
        json.dump(digests, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(OUT, "ref_topology.npz"), **arrays)
    print(len(digests), "cases,", len(arrays), "arrays")
