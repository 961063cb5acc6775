"""bvhNN_optimize / bvh_optimize_nodes = the reference's ReinsertionOptimizer (reinsertion_optimizer.h:27-30,88-267).

A tree built by the UNMODIFIED reference C library is optimised twice: by the reference's own bvhNN_optimize and by this
library (bvh_optimize_nodes on the same node array, and — for the 2-D suffixes, which need no GPU — bvh2f_load +
bvh2f_optimize + bvh2f_save).  The results must be identical node for node, serial and multi-threaded, and the pass must
actually lower the tree's SAH cost.  The reference's side is stored (tests/golden/make_ref_digests.py): the topology of
the tree it builds, from which tests/helpers.py tree_blob rebuilds its exact file, and digests of what its pass returns."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.helpers import digest, ref_digests, tree_blob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OURS = os.path.join(ROOT, "bvh_b200", "libbvh_c.so")
libc = C.CDLL(None)
libc.fopen.restype = C.c_void_p
libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
libc.fclose.argtypes = [C.c_void_p]


def bind(lib, s):
    f = lambda name: getattr(lib, f"bvh{s}_{name}")
    f("build").restype = C.c_void_p
    f("build").argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    f("load").restype = C.c_void_p; f("load").argtypes = [C.c_void_p]
    f("save").argtypes = [C.c_void_p, C.c_void_p]
    f("destroy").argtypes = [C.c_void_p]
    f("optimize").argtypes = [C.c_void_p, C.c_void_p]
    lib.bvh_thread_pool_create.restype = C.c_void_p
    lib.bvh_thread_pool_create.argtypes = [C.c_size_t]
    lib.bvh_thread_pool_destroy.argtypes = [C.c_void_p]
    return f


def save_bytes(f, bvh, path):
    fp = libc.fopen(str(path).encode(), b"wb"); f("save")(bvh, fp); libc.fclose(fp)
    return open(path, "rb").read()


def load_file(f, path):
    fp = libc.fopen(str(path).encode(), b"rb"); h = f("load")(fp); libc.fclose(fp)
    return h


def parse(blob, dim, dtype):
    """Serialised tree (bvh.h:220-242) -> (node records as a structured array, prim ids)."""
    it = np.dtype(np.uint32 if dtype == np.float32 else np.uint64)
    node_count, prim_count = (int(x) for x in np.frombuffer(blob, it, 2))
    node_dt = np.dtype([("bounds", dtype, 2 * dim), ("index", it)])
    assert node_dt.itemsize == (2 * dim + 1) * it.itemsize
    nodes = np.frombuffer(blob, node_dt, node_count, 2 * it.itemsize).copy()
    ids = np.frombuffer(blob, it, prim_count, 2 * it.itemsize + node_count * node_dt.itemsize).copy()
    return nodes, ids


def sah_cost(nodes, dim):
    b = nodes["bounds"].astype(np.float64)
    d = b[:, 1::2] - b[:, 0::2]
    area = (d[:, 0] + d[:, 1]) * d[:, 2] + d[:, 0] * d[:, 1] if dim == 3 else d[:, 0] + d[:, 1]
    count = (nodes["index"] & 15).astype(np.float64)
    return float(np.where(count > 0, area * count, area).sum() / area[0])


def scene(dim, n, dtype, seed):
    rng = np.random.default_rng(seed)
    c = rng.random((n, dim))
    c[: n // 3] = 0.5 + 0.02 * rng.standard_normal((n // 3, dim))        # a dense cluster: uneven areas, real reinsertions
    ext = rng.random((n, dim)) * rng.choice([0.002, 0.02, 0.2], size=(n, 1))
    lo, hi = (c - ext).astype(dtype), (c + ext).astype(dtype)
    centers = ((lo.astype(np.float64) + hi) * 0.5).astype(dtype)
    return np.ascontiguousarray(np.concatenate([lo, hi], axis=1)), np.ascontiguousarray(centers)


@pytest.mark.parametrize("s,dim,dtype", [("3f", 3, np.float32), ("3d", 3, np.float64), ("2f", 2, np.float32), ("2d", 2, np.float64)])
@pytest.mark.parametrize("n", [300, 3000])
def test_optimize_nodes_equals_the_reference(tmp_path, s, dim, dtype, n):
    ours = C.CDLL(OURS)
    boxes, centers = scene(dim, n, dtype, 7 + n)
    ref = ref_digests(f"optimize/{s}/{n}")
    with np.load(os.path.join(ROOT, "tests", "golden", "ref_topology.npz")) as g:
        before = tree_blob(g[f"optimize/{s}/{n}/index"], g[f"optimize/{s}/{n}/prim_ids"], boxes, dim)
    assert digest(before) == ref["before"], "the stored topology no longer gives the reference's tree"
    if n >= 3000:
        assert ref["after"] != ref["before"], "the scene must give the optimizer something to do"
    (tmp_path / "before.bin").write_bytes(before)

    nodes, ids = parse(before, dim, dtype)
    ours.bvh_optimize_nodes.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_double, C.c_size_t, C.c_size_t]
    ours.bvh_last_error.restype = C.c_char_p
    for threads in (1, 5):
        mine = nodes.copy()
        rc = ours.bvh_optimize_nodes(mine.ctypes.data, mine.shape[0], dim, dtype == np.float64, 0.05, 3, threads)
        assert rc == 0, ours.bvh_last_error()
        assert digest(mine) == ref["after_nodes"], f"{threads} thread(s): tree differs from the reference's optimised tree"
    assert digest(ids) == ref["after_prim_ids"]                   # the pass never touches the primitive order
    assert sah_cost(mine, dim) <= sah_cost(nodes, dim)            # `mine` is now bit for bit the reference's result
    if n >= 3000:
        assert sah_cost(mine, dim) < sah_cost(nodes, dim)

    if dim == 2:                                                  # the host-only suffixes: through load / optimize / save
        of = bind(ours, s)
        h = load_file(of, tmp_path / "before.bin")
        opool = ours.bvh_thread_pool_create(3)
        of("optimize")(opool, h)
        ours.bvh_thread_pool_destroy(opool)
        assert digest(save_bytes(of, h, tmp_path / "after_ours.bin")) == ref["after"]
        of("destroy")(h)


def test_optimize_rejects_a_broken_tree():
    ours = C.CDLL(OURS)
    ours.bvh_optimize_nodes.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_double, C.c_size_t, C.c_size_t]
    ours.bvh_last_error.restype = C.c_char_p
    node_dt = np.dtype([("bounds", np.float32, 6), ("index", np.uint32)])
    nodes = np.zeros(5, node_dt)
    nodes["index"] = [1 << 4, 3 << 4, 1, 1, 1]                   # root -> (1, 2); node 1 -> (3, 4): fine
    assert ours.bvh_optimize_nodes(nodes.ctypes.data, 5, 3, 0, 0.05, 3, 1) == 0
    nodes["index"][1] = 9 << 4                                    # child index out of range
    assert ours.bvh_optimize_nodes(nodes.ctypes.data, 5, 3, 0, 0.05, 3, 1) != 0
    assert b"well-formed" in ours.bvh_last_error()
    nodes["index"][1] = 1 << 4                                    # a cycle: node 1 claims the root's children
    assert ours.bvh_optimize_nodes(nodes.ctypes.data, 5, 3, 0, 0.05, 3, 1) != 0
    assert ours.bvh_optimize_nodes(None, 5, 3, 0, 0.05, 3, 1) != 0
    assert ours.bvh_optimize_nodes(nodes.ctypes.data, 5, 4, 0, 0.05, 3, 1) != 0
