"""2-D suffixes of the C ABI (bvh2f / bvh2d, reference c_api/bvh.cpp:7-25).

CPU part: the file of a tree built and saved by the UNMODIFIED reference C library (rebuilt from its stored topology,
tests/golden/make_ref_digests.py) is loaded through our library; node accessors, per-ray callback traversal (all four
variants), refit and save must then agree with the reference's stored answers bit for bit.  GPU part: bvh2f_build /
bvh2d_build (the LBVH pipeline on boxes lifted to z = 0) produce a valid tree whose traversal finds the brute-force
answer."""
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


def slab(dtype, ray, box, tmax):
    """Entry distance of a 2-D ray into a box (None on a miss); plain python floats, result rounded to dtype."""
    t0, t1 = ray[4], tmax
    for k in range(2):
        d = ray[2 + k]
        if d == 0:
            if not (box[k] <= ray[k] <= box[2 + k]): return None
            continue
        a, b = (box[k] - ray[k]) / d, (box[2 + k] - ray[k]) / d
        t0, t1 = max(t0, min(a, b)), min(t1, max(a, b))
    return dtype(t0) if t0 <= t1 else None


class Api2:
    """ctypes view of the 2-D entry points of one library (ours or the reference's: same ABI)."""

    def __init__(self, path, s):
        self.lib, self.s = C.CDLL(path), s
        self.ct = C.c_float if s == "2f" else C.c_double
        self.dtype = np.float32 if s == "2f" else np.float64
        ct = self.ct

        class Vec(C.Structure): _fields_ = [("x", ct), ("y", ct)]
        class BBox(C.Structure): _fields_ = [("min", Vec), ("max", Vec)]
        class Ray(C.Structure): _fields_ = [("org", Vec), ("dir", Vec), ("tmin", ct), ("tmax", ct)]
        self.FN = C.CFUNCTYPE(C.c_bool, C.c_void_p, C.POINTER(ct), C.c_size_t, C.c_size_t)
        class Callback(C.Structure): _fields_ = [("user_data", C.c_void_p), ("user_fn", self.FN)]
        self.Vec, self.BBox, self.Ray, self.Callback = Vec, BBox, Ray, Callback
        f = lambda name: getattr(self.lib, f"bvh{s}_{name}")
        g = lambda name: getattr(self.lib, f"bvh_node{s}_{name}")
        f("build").restype = C.c_void_p
        f("build").argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        f("load").restype = C.c_void_p; f("load").argtypes = [C.c_void_p]
        f("save").argtypes = [C.c_void_p, C.c_void_p]
        f("destroy").argtypes = [C.c_void_p]
        f("get_node").restype = C.c_void_p; f("get_node").argtypes = [C.c_void_p, C.c_size_t]
        for name in ("get_prim_count", "get_node_count"):
            f(name).restype = C.c_size_t; f(name).argtypes = [C.c_void_p]
        f("get_prim_id").restype = C.c_size_t; f("get_prim_id").argtypes = [C.c_void_p, C.c_size_t]
        for name in ("refit", "append_node", "remove_last_node"): f(name).argtypes = [C.c_void_p]
        for name in ("intersect_ray", "intersect_ray_any", "intersect_ray_robust", "intersect_ray_any_robust"):
            f(name).argtypes = [C.c_void_p, C.POINTER(Ray), C.POINTER(Callback)]
        g("is_leaf").restype = C.c_bool; g("is_leaf").argtypes = [C.c_void_p]
        for name in ("get_prim_count", "get_first_id"):
            g(name).restype = C.c_size_t; g(name).argtypes = [C.c_void_p]
        for name in ("set_prim_count", "set_first_id"): g(name).argtypes = [C.c_void_p, C.c_size_t]
        g("get_bbox").restype = BBox; g("get_bbox").argtypes = [C.c_void_p]
        g("set_bbox").argtypes = [C.c_void_p, C.POINTER(BBox)]
        self.f, self.g = f, g

    def build(self, boxes, centers):
        boxes = np.ascontiguousarray(boxes, self.dtype); centers = np.ascontiguousarray(centers, self.dtype)
        return self.f("build")(None, boxes.ctypes.data, centers.ctypes.data, boxes.shape[0], None)

    def save(self, bvh, path):
        fp = libc.fopen(path.encode(), b"wb"); self.f("save")(bvh, fp); libc.fclose(fp)

    def load(self, path):
        fp = libc.fopen(path.encode(), b"rb"); h = self.f("load")(fp); libc.fclose(fp); return h

    def nodes(self, bvh):
        out = []
        for i in range(self.f("get_node_count")(bvh)):
            nd = self.f("get_node")(bvh, i)
            b = self.g("get_bbox")(nd)
            out.append((b.min.x, b.min.y, b.max.x, b.max.y, self.g("is_leaf")(nd), self.g("get_first_id")(nd), self.g("get_prim_count")(nd)))
        return out

    def prim_ids(self, bvh):
        return [self.f("get_prim_id")(bvh, i) for i in range(self.f("get_prim_count")(bvh))]

    def trace(self, bvh, rays, boxes, ids, variant="intersect_ray"):
        """Closest (or any) hit of 2-D rays against the primitive BOXES, via the leaf callback.  Returns
        (original prim id or -1, t, number of callback invocations) per ray."""
        results = []
        state = {}
        def leaf(_, t, begin, end):
            hit = False
            state["calls"] += 1
            for i in range(begin, end):
                tt = slab(self.dtype, state["ray"], [float(x) for x in boxes[ids[i]]], float(t[0]))
                if tt is not None and tt <= t[0]:
                    t[0] = tt; state["id"] = ids[i]; state["t"] = float(tt); hit = True
            return hit
        cb = self.Callback(None, self.FN(leaf))
        for r in rays:
            state.update(ray=[float(x) for x in r], id=-1, calls=0, t=None)
            ray = self.Ray(self.Vec(r[0], r[1]), self.Vec(r[2], r[3]), r[4], r[5])
            self.f(variant)(bvh, C.byref(ray), C.byref(cb))
            results.append((state["id"], state["t"], state["calls"]))
        return results


def scene2(n, seed, dtype):
    rng = np.random.default_rng(seed)
    c = rng.random((n, 2))
    half = rng.random((n, 2)) * (0.6 / np.sqrt(n))
    boxes = np.concatenate([c - half, c + half], axis=1).astype(dtype)           # min.x min.y max.x max.y
    centers = ((boxes[:, :2].astype(np.float64) + boxes[:, 2:]) * 0.5).astype(dtype)
    m = 200
    org = rng.random((m, 2)) * 1.4 - 0.2
    ang = rng.random(m) * 2 * np.pi
    rays = np.concatenate([org, np.cos(ang)[:, None], np.sin(ang)[:, None], np.zeros((m, 1)), np.full((m, 1), 10.0)], axis=1).astype(dtype)
    rays[:8, 2] = 0          # axis-parallel rays (division by zero in the slab test: safe_inverse / robust)
    rays[8:16, 3] = 0
    return boxes, centers, rays


@pytest.mark.parametrize("s", ["2f", "2d"])
def test_loaded_reference_tree_behaves_like_the_reference(tmp_path, s):
    ours = Api2(OURS, s)
    want = ref_digests(f"c_abi_2d/{s}")
    boxes, centers, rays = scene2(700, 3, ours.dtype)
    with np.load(os.path.join(ROOT, "tests", "golden", "ref_topology.npz")) as g:
        stored = {k[len(f"c_abi_2d/{s}/"):]: g[k] for k in g.files if k.startswith(f"c_abi_2d/{s}/")}
    blob = tree_blob(stored["index"], stored["prim_ids"], boxes, 2)
    assert digest(blob) == want["blob"]
    path = str(tmp_path / f"tree_{s}.bin")
    open(path, "wb").write(blob)
    ob = ours.load(path)
    assert ours.f("get_node_count")(ob) == stored["index"].shape[0] > 1
    assert digest(np.array(ours.nodes(ob), np.float64)) == want["nodes"]
    ids = [int(i) for i in stored["prim_ids"]]
    assert ours.prim_ids(ob) == ids and sorted(ids) == list(range(700))
    for variant in ("intersect_ray", "intersect_ray_any", "intersect_ray_robust", "intersect_ray_any_robust"):
        got = ours.trace(ob, rays, boxes, ids, variant)
        ref = [(int(i), None if np.isnan(t) else float(t), int(c))
               for i, t, c in zip(*(stored[f"{variant}/{k}"] for k in ("id", "t", "calls")))]
        assert got == ref, variant                         # same hits AND the same sequence of leaf visits
        assert sum(1 for g in got if g[0] >= 0) > 50

    # grow every leaf box, refit, and compare again; then save and compare the bytes
    for i in range(ours.f("get_node_count")(ob)):
        nd = ours.f("get_node")(ob, i)
        if ours.g("is_leaf")(nd):
            b = ours.g("get_bbox")(nd)
            b.max.x += 0.25; b.min.y -= 0.125
            ours.g("set_bbox")(nd, C.byref(b))
    ours.f("refit")(ob)
    assert digest(np.array(ours.nodes(ob), np.float64)) == want["refit_nodes"]
    p1 = str(tmp_path / "a.bin")
    ours.save(ob, p1)
    assert digest(open(p1, "rb").read()) == want["refit_blob"]

    # node editing entry points
    nd = ours.f("get_node")(ob, 1)
    ours.g("set_first_id")(nd, 12345); ours.g("set_prim_count")(nd, 3)
    assert ours.g("get_first_id")(nd) == 12345 and ours.g("get_prim_count")(nd) == 3 and ours.g("is_leaf")(nd)
    count = ours.f("get_node_count")(ob)
    ours.f("append_node")(ob); assert ours.f("get_node_count")(ob) == count + 1
    ours.f("remove_last_node")(ob); assert ours.f("get_node_count")(ob) == count
    ours.f("destroy")(ob)


@pytest.mark.gpu
@pytest.mark.parametrize("s,n", [("2f", 1), ("2f", 2), ("2f", 3000), ("2d", 1500)])
def test_gpu_build_2d(tmp_path, s, n):
    ours = Api2(OURS, s)
    boxes, centers, rays = scene2(n, 11, ours.dtype)
    bvh = ours.build(boxes, centers)
    assert bvh, "bvh%s_build failed" % s
    nodes, ids = ours.nodes(bvh), ours.prim_ids(bvh)
    assert sorted(ids) == list(range(n))
    covered = np.zeros(n, bool)
    for i, (x0, y0, x1, y1, leaf, first, count) in enumerate(nodes):
        if leaf:
            assert 1 <= count <= 8
            for k in range(first, first + count):
                assert not covered[k]; covered[k] = True
                b = boxes[ids[k]]
                assert x0 <= b[0] and y0 <= b[1] and x1 >= b[2] and y1 >= b[3]
        else:
            assert first % 2 == 1 and first + 1 < len(nodes)
            for c in (nodes[first], nodes[first + 1]):
                assert x0 <= c[0] and y0 <= c[1] and x1 >= c[2] and y1 >= c[3]
    assert covered.all()
    got = ours.trace(bvh, rays, boxes, ids, "intersect_ray_robust")
    hits = 0
    for r, g in zip(rays, got):                            # brute force over all primitives, same arithmetic
        ray, best = [float(x) for x in r], float(r[5])
        found = False
        for k in range(n):
            tt = slab(ours.dtype, ray, [float(x) for x in boxes[k]], best)
            if tt is not None and tt <= best: best, found = float(tt), True
        assert (g[0] >= 0) == found
        if found: assert g[1] == best; hits += 1
    assert n < 100 or hits > 50
    # same tree through save / load gives the same answers
    path = str(tmp_path / "t.bin")
    ours.save(bvh, path)
    again = ours.load(path)
    assert ours.nodes(again) == nodes and ours.trace(again, rays, boxes, ids, "intersect_ray_robust") == got
    ours.f("destroy")(again); ours.f("destroy")(bvh)
