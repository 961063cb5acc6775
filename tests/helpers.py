"""Test helpers: the host emulation of the device code (tests/host_emul.cpp) and comparison utilities."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 0xFFFFFFFF
P = C.c_void_p


def _ptr(a):
    return None if a is None else a.ctypes.data_as(P)


def aligned_zeros(shape, dtype, align=128):
    """numpy zeros whose data pointer is `align`-byte aligned (the device structs are alignas(32/64) and
    g++ emits aligned vector moves for them; cudaMalloc gives 256-byte alignment on the GPU)."""
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    raw = np.zeros(count * dtype.itemsize + align, np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + count * dtype.itemsize].view(dtype).reshape(shape)


def build_host_emul() -> str:
    src = os.path.join(ROOT, "tests", "host_emul.cpp")
    out_dir = os.path.join(ROOT, "tests", "_build")
    out = os.path.join(out_dir, "libhost_emul.so")
    csrc = os.path.join(ROOT, "bvh_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("core.cuh", "build_core.cuh", "traverse_core.cuh", "treelet_warp.cuh", "wide_bvh.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC",
                               "-shared", "-x", "c++", "-I", csrc, src, "-o", out])
    return out


class HostEmul:
    """Runs the per-thread device functions sequentially on the CPU (logic check without a GPU)."""

    def __init__(self):
        self.lib = L = C.CDLL(build_host_emul())
        for s in ("3f", "3d"):
            getattr(L, f"emul_build{s}").restype = C.c_uint32
            getattr(L, f"emul_build{s}").argtypes = [P, P, P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, P, P, P, P]
            getattr(L, f"emul_compact{s}").restype = C.c_size_t
            getattr(L, f"emul_compact{s}").argtypes = [P, C.c_size_t, P, P, C.c_size_t]
            getattr(L, f"emul_trace{s}").argtypes = [P, P, P, P, C.c_size_t, C.c_uint, P, P, P, P, P]
            getattr(L, f"emul_from_reference{s}").argtypes = [P, P, C.c_size_t, P]
            getattr(L, f"emul_precompute{s}").argtypes = [P, P, C.c_size_t, P]
        L.emul_wide_build.restype = C.c_size_t
        L.emul_wide_build.argtypes = [P, P, C.c_size_t, P]
        L.emul_wide_trace.argtypes = [P, P, P, P, C.c_size_t, C.c_uint, P, P, P, P, P]
        L.emul_set_block.argtypes = [C.c_int, C.c_int]
        L.emul_set_treelets.argtypes = [C.c_int]
        L.emul_last_treelet_count.restype = C.c_int
        L.emul_last_node_slots.restype = C.c_size_t
        L.emul_morton30.restype = C.c_uint32
        L.emul_morton30.argtypes = [C.c_uint32] * 3
        L.emul_morton63.restype = C.c_uint64
        L.emul_morton63.argtypes = [C.c_uint64] * 3

    @staticmethod
    def _s(dtype):
        return "3f" if np.dtype(dtype) == np.float32 else "3d"

    def build(self, tris=None, bboxes=None, centers=None, min_leaf=1, max_leaf=8, morton_bits=30, quality=None):
        """``quality`` mirrors the library: "low" = plain LBVH, "medium" / "high" = + SAH treelet pass; None keeps
        whatever set_treelets() selected."""
        if quality is not None:
            self.set_treelets(quality != "low")
            try:
                return self.build(tris, bboxes, centers, min_leaf, max_leaf, morton_bits)
            finally:
                self.set_treelets(False)
        src = tris if tris is not None else bboxes
        dtype, n = src.dtype, src.shape[0]
        s = self._s(dtype)
        words = 8  # a device node is 8 scalars wide (6 bounds + index + pad) for both float and double
        nodes = aligned_zeros((2 * n, words), dtype)
        ids = np.zeros(n, np.uint32)
        dtris = aligned_zeros((n, 16), dtype) if tris is not None else None   # room for the padded record form (BVH_TRI_PAD)
        depth = C.c_uint32(0)
        getattr(self.lib, f"emul_build{s}")(_ptr(tris), _ptr(bboxes), _ptr(centers), n, min_leaf, max_leaf, morton_bits,
                                            _ptr(nodes), _ptr(ids), _ptr(dtris), C.byref(depth))
        # the emulation compacts like the device build: `slots` dense device slots (slot 0 padding, slot 1 the root)
        return dict(nodes=nodes, prim_ids=ids, tris=dtris, depth=depth.value, dtype=dtype, n=n, slots=self.lib.emul_last_node_slots())

    def set_treelets(self, on, reversed_phases: bool = False):
        """Experimental second build pass: SAH rebuild of the LBVH's bottom subtrees (treelet_warp.cuh);
        ``reversed_phases`` runs the iterations of every phase in descending order (hazard check)."""
        self.lib.emul_set_treelets((2 if reversed_phases else 1) if on else 0)

    def set_block(self, leaves=0, order=0):
        """0 leaves: every merge through the global flags; else the device kernel's block-local first phase."""
        self.lib.emul_set_block(leaves, order)

    def compact(self, tree):
        n, dtype = tree["n"], tree["dtype"]
        bounds = np.zeros((2 * n, 6), dtype)
        index_values = np.zeros(2 * n, np.uint64)
        cnt = getattr(self.lib, f"emul_compact{self._s(dtype)}")(_ptr(tree["nodes"]), tree["slots"], _ptr(bounds), _ptr(index_values), 2 * n)
        return bounds[:cnt].copy(), index_values[:cnt].copy()

    def from_reference(self, bounds, index_values, prim_ids, tris):
        """Device-layout copy of a reference-layout tree (what c_api.cu upload_mirror produces)."""
        dtype = bounds.dtype
        n_nodes = bounds.shape[0]
        nodes = aligned_zeros((n_nodes + 1, 8), dtype)
        s = self._s(dtype)
        getattr(self.lib, f"emul_from_reference{s}")(_ptr(np.ascontiguousarray(bounds)),
                                                    _ptr(np.ascontiguousarray(index_values, dtype=np.uint64)), n_nodes, _ptr(nodes))
        ids = np.ascontiguousarray(prim_ids, dtype=np.uint32)
        dtris = aligned_zeros((ids.shape[0], 16), dtype)
        getattr(self.lib, f"emul_precompute{s}")(_ptr(np.ascontiguousarray(tris)), _ptr(ids), ids.shape[0], _ptr(dtris))
        return dict(nodes=nodes, prim_ids=ids, tris=dtris, depth=None, dtype=dtype, n=ids.shape[0], slots=n_nodes + 1)

    def wide_build(self, tree):
        """Collapse the (float) binary tree into the compressed 4-wide tree; returns (wide nodes, levels)."""
        n = tree["n"]
        wide = aligned_zeros((max(n, 1), 16), np.uint32)
        levels = C.c_uint32(0)
        count = self.lib.emul_wide_build(_ptr(tree["nodes"]), _ptr(wide), wide.shape[0], C.byref(levels))
        assert count <= wide.shape[0]
        return wide[:count], levels.value

    def wide_trace(self, tree, wide, rays, flags):
        rays = np.ascontiguousarray(rays, dtype=np.float32)
        m = rays.shape[0]
        ids = np.zeros(m, np.uint32)
        t, u, v = (np.zeros(m, np.float32) for _ in range(3))
        steps = np.zeros(m, np.uint32)
        self.lib.emul_wide_trace(_ptr(wide), _ptr(tree["tris"]), _ptr(tree["prim_ids"]), _ptr(rays), m, flags,
                                 _ptr(ids), _ptr(t), _ptr(u), _ptr(v), _ptr(steps))
        return ids, t, u, v, steps

    def trace(self, tree, rays, flags):
        dtype = tree["dtype"]
        rays = np.ascontiguousarray(rays, dtype=dtype)
        m = rays.shape[0]
        ids = np.zeros(m, np.uint32)
        t, u, v = (np.zeros(m, dtype) for _ in range(3))
        st = np.zeros((m, 3), np.uint32)
        getattr(self.lib, f"emul_trace{self._s(dtype)}")(_ptr(tree["nodes"]), _ptr(tree["tris"]), _ptr(tree["prim_ids"]),
                                                       _ptr(rays), m, flags, _ptr(ids), _ptr(t), _ptr(u), _ptr(v), _ptr(st))
        return ids, t, u, v, st


def assert_hits_equal(got, want, what=""):
    """Bit-exact comparison of (ids, t, u, v) tuples."""
    names = ("ids", "t", "u", "v")
    for name, a, b in zip(names, got, want):
        a, b = np.asarray(a), np.asarray(b)
        if a.dtype.kind == "f":
            same = a.view(np.uint32 if a.dtype == np.float32 else np.uint64) == b.view(np.uint32 if b.dtype == np.float32 else np.uint64)
        else:
            same = a.astype(np.uint64) == b.astype(np.uint64)
        assert same.all(), f"{what}: {name} differs at {np.nonzero(~same)[0][:8]} ({(~same).sum()} of {same.size})"


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and bytes (bytes objects count as uint8 arrays): equal digests mean
    bit-identical arrays, so a stored digest pins an output of the reference as strictly as the output itself."""
    a = np.ascontiguousarray(np.frombuffer(a, np.uint8) if isinstance(a, bytes) else a)
    return hashlib.sha256(a.dtype.str.encode() + repr(a.shape).encode() + a.tobytes()).hexdigest()


def ref_digests(key):
    """Digests of the reference's outputs for one test case (tests/golden/make_ref_digests.py)."""
    with open(os.path.join(ROOT, "tests", "golden", "ref_digests.json")) as f:
        return json.load(f)[key]


def tree_blob(index, prim_ids, boxes, dim):
    """The reference's file format (bvh.h serialize) of the tree with the given topology over `boxes` ([n, 2*dim]: mins then
    maxes): every node box is the exact union of the primitive boxes below it, as the reference's builders make them.
    Index words and prim ids are 32-bit for float trees and 64-bit for double trees; children follow their parent."""
    dtype = boxes.dtype
    it = np.dtype(np.uint32 if dtype == np.float32 else np.uint64)
    index = np.asarray(index, np.uint64)
    prim_ids = np.asarray(prim_ids, np.int64)
    lo, hi = boxes[:, :dim], boxes[:, dim:]
    bounds = np.empty((index.shape[0], 2 * dim), dtype)
    for i in range(index.shape[0] - 1, -1, -1):
        first, count = int(index[i] >> np.uint64(4)), int(index[i] & np.uint64(15))
        if count:
            ids = prim_ids[first:first + count]
            bounds[i, 0::2], bounds[i, 1::2] = lo[ids].min(axis=0), hi[ids].max(axis=0)
        else:
            assert first > i, "a child precedes its parent"
            bounds[i, 0::2] = np.minimum(bounds[first, 0::2], bounds[first + 1, 0::2])
            bounds[i, 1::2] = np.maximum(bounds[first, 1::2], bounds[first + 1, 1::2])
    nodes = np.zeros(index.shape[0], [("bounds", dtype, 2 * dim), ("index", it)])
    nodes["bounds"], nodes["index"] = bounds, index
    return np.array([index.shape[0], prim_ids.shape[0]], it).tobytes() + nodes.tobytes() + prim_ids.astype(it).tobytes()


def hits_tuple(hits):
    """structured bvh_hit array -> (ids, t, u, v) with 32-bit ids"""
    return hits["prim_id"].astype(np.uint32), hits["t"], hits["u"], hits["v"]


def assert_hits_conservative(got, want, tris, rays, oracle, what="", max_fraction=1e-5):
    """The default traversal path (compressed 4-wide tree) against an exact binary traversal of the reference's
    algorithm (`want` = (ids, t, u, v)).  The wide boxes enclose the binary ones, the triangle test and the
    tie-break are the same, so the results are identical except where the binary traversal itself misses a true hit
    because the reference's FAST slab test is not watertight (a hit point exactly on a box face).  There — and only
    there — the wide path may report a closer hit, or the same distance with a lower id, and that hit must be real."""
    g = hits_tuple(got) if not isinstance(got, tuple) else got
    bits = lambda a: np.asarray(a).view(np.uint32 if np.asarray(a).dtype.itemsize == 4 else np.uint64)
    same = (np.asarray(g[0]).astype(np.uint64) == np.asarray(want[0]).astype(np.uint64))
    for k in (1, 2, 3):
        same &= bits(g[k]) == bits(want[k])
    bad = np.nonzero(~same)[0]
    assert bad.size <= max(2, max_fraction * same.size), f"{what}: {bad.size} of {same.size} rays differ"
    for i in bad:
        assert g[0][i] != INVALID, f"{what}: ray {i} lost its hit"
        assert g[1][i] < want[1][i] or (g[1][i] == want[1][i] and g[0][i] < want[0][i]), f"{what}: ray {i} is not closer"
        one = oracle.brute_force(tris[int(g[0][i]):int(g[0][i]) + 1], rays[i:i + 1])
        assert one[0][0] == 0 and one[1][0] == g[1][i] and one[2][0] == g[2][i] and one[3][0] == g[3][i], f"{what}: ray {i}: not a real hit"
