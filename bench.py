#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json measured on B200(s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c3|c4|c5] [--mesh soup|grid]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default (`--config c2`, BASELINE.json configs[1]): a step is one pass of the batched closest-hit traversal
over 10M coherent primary rays (3163 x 3163 pinhole camera, reference test/benchmark.cpp:340-358) against a
1M-triangle synthetic mesh; with N GPUs every rank traces its own 10M-ray shard of an N x 10M batch (BVH
replicated, weak scaling) and the 16-byte hit records are gathered on every rank inside the traversal kernel
(peer stores over NVLink) or by NCCL.  `value` is whole-job Mrays/s with rays resident in HBM; `build` reports
the LBVH build rate of the same mesh (Mtris/s) timed in the same run; `e2e` is the same metric through the
C ABI with pinned HOST buffers (H2D of the rays and D2H of the hits inside the timed region).

Other BASELINE configs (same JSON shape): c3 = 10M incoherent AO-style rays, any-hit; c4 = 10M triangles,
100M primary rays sharded over the ranks (strong scaling, 63-bit Morton keys); c5 = double precision,
100K triangles, 1M rays.

`--impl reference` times the reference's own CPU implementation (oracle/_ref = the unmodified reference
compiled in place; the plain-C oracle port when that is absent) on the SAME rays with every usable host
thread, and prints the same JSON line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bvh_b200 import scenes  # noqa: E402

FALLBACK_HBM_GBS = 6650.0        # /opt/skills/guides/B200_PROFILING.md fallback

# BASELINE.json configs[1..4].  img: the camera is img x img primary rays; count: incoherent rays.
CONFIGS = {
    "c2": dict(tris=1_000_000, img=3163, dtype="f32", any_hit=False, scaling="weak",
               metric="primary closest-hit rays per second"),
    "c3": dict(tris=1_000_000, count=10_000_000, dtype="f32", any_hit=True, scaling="weak",
               metric="incoherent any-hit (AO) rays per second"),
    "c4": dict(tris=10_000_000, img=10_000, dtype="f32", any_hit=False, scaling="strong",
               metric="primary closest-hit rays per second"),
    "c5": dict(tris=100_000, img=1000, dtype="f64", any_hit=False, scaling="weak",
               metric="primary closest-hit rays per second"),
}
AUTO_DIRECT_MAX_RANKS = 4         # --gather auto: per-record peer stores up to this many ranks, staged bulk copies beyond
C4_CPU_ROW_STRIDE = 10           # the CPU arm of c4 traces every 10th image row (10M of the 100M rays)
DUMP_MAX_RAYS = 1 << 20          # --dump-outputs: at most this many hit records (28 MB in f32, 40 MB in f64)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--mesh", default="soup", choices=["soup", "grid"])
    ap.add_argument("--quality", default=None, choices=["low", "medium", "high"],
                    help="DefaultBuilder::Quality passed to the build (default: the library default, High)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--kernel", default="auto", choices=["auto", "persistent", "tma", "wide", "simple"],
                    help="auto: the library's default choice for the flags of the config")
    ap.add_argument("--chunks", type=int, default=4, help="NCCL gather chunks per step when N > 1 and --gather nccl")
    ap.add_argument("--gather", default="auto", choices=["auto", "multicast", "multicast_staged", "peer", "direct", "nccl"],
                    help="N > 1: fused gather inside the traversal kernel — peer (= auto): a warp stages 32 records in shared memory and "
                         "bulk-copies them to every rank; direct: one 16-byte store per record and rank; multicast: one multimem.st per "
                         "record — or NCCL all-gather")
    ap.add_argument("--sort-rays", action="store_true", help="BVH_SORT_RAYS: traverse the batch in the Morton order of the ray origins")
    ap.add_argument("--no-numa", action="store_true", help="N > 1: do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the hit records of the last timed step as DIR/<field>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path")
    return args


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def usable_cpus():
    """CPUs this process may actually use: the affinity mask, capped by the cgroup CPU quota (a pool of
    hardware_concurrency threads on a host whose cgroup grants fewer CPUs oversubscribes and thrashes)."""
    try:
        affinity = len(os.sched_getaffinity(0))
    except Exception:
        affinity = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    usable = affinity if quota is None else max(1, min(affinity, int(quota)))
    return {"usable": usable, "affinity": affinity, "cgroup_quota": quota, "hardware": os.cpu_count()}


def gather_candidates(world: int, requested: str) -> list:
    """Delivery forms of the fused gather to try, in order; an empty list means the NCCL path.  `auto` follows the
    measurements of DESIGN.md §7: two ranks — one multimem store per record; up to AUTO_DIRECT_MAX_RANKS — one peer store
    per record and rank; beyond — warp-staged bulk copies, to the multicast address when the fabric has one."""
    if world == 1 or requested == "nccl":
        return []
    if requested != "auto":
        return [requested]
    if world == 2:
        return ["multicast", "direct", "peer"]
    if world <= AUTO_DIRECT_MAX_RANKS:
        return ["direct", "peer"]
    return ["multicast_staged", "peer", "direct"]


def bind_to_gpu_numa_node(local_rank: int):
    """Multi-rank runs: pin this rank (and therefore the first-touch placement of its pinned host buffers)
    to the NUMA node its GPU hangs off.  Eight ranks streaming 70 GB/s each through whatever socket the
    scheduler put them on is what collapsed the 8-GPU e2e number in round 1."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        sysfs = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node"
        node = int(open(sysfs).read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception as exc:
        return {"error": f"{type(exc).__name__}: {exc}"}


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (NVML; nvidia-smi as a fallback)."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag = index, threading.Event()
        self.sm, self.sm_max, self.reasons = [], None, set()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def sample(self):
        if self.nvml is not None:
            n = self.nvml
            self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
            try:
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:
                mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            for name, bit in self.REASONS:
                if mask & bit:
                    self.reasons.add(name)
            return
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        self.sm.append(float(f[0]))
        self.sm_max = float(f[1])
        for (name, _), v in zip(self.REASONS, f[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self.sample()
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no samples"], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def np_dtype(cfg):
    return np.float32 if cfg["dtype"] == "f32" else np.float64


def make_tris(cfg, kind):
    return scenes.make_mesh(kind, cfg["tris"], dtype=np_dtype(cfg))


def make_rays(cfg, kind, tris, rank=0, world=1, row_stride=1):
    """This rank's rays.  weak scaling: the full batch of the config, made distinct per rank (sub-pixel camera
    offset rank/world; another seed for the incoherent rays) so that the global batch is world x the config's
    rays of one distribution.  strong scaling (c4): this rank's band of image rows."""
    dt = np_dtype(cfg)
    if "count" in cfg:
        return scenes.incoherent_rays(tris, cfg["count"], seed=12345 + rank)
    img = cfg["img"]
    if cfg["scaling"] == "strong":
        assert img % world == 0, "the c4 camera has 10000 rows: use 1, 2, 4, 5, 8 or 10 ranks"
        y0, y1 = rank * img // world, (rank + 1) * img // world
        rays = scenes.make_primary(kind, img, img, dtype=dt, y_begin=y0, y_end=y1)
    else:
        rays = scenes.make_primary(kind, img, img, dtype=dt, pixel_offset=rank / world)
    if row_stride > 1:
        rays = np.ascontiguousarray(rays.reshape(-1, img, 8)[::row_stride].reshape(-1, 8))
    return rays


def workload_text(cfg, kind, name):
    rays = (f"{cfg['count']} incoherent AO-style rays (tmax 0.25), any-hit" if "count" in cfg else
            f"{cfg['img']}x{cfg['img']} = {cfg['img'] ** 2} coherent primary rays, closest-hit")
    per = "sharded over the ranks" if cfg["scaling"] == "strong" else "per GPU"
    return f"{name}: {kind}-{cfg['tris']} triangles, {rays} {per}, {cfg['dtype']}"


def bytes_per_ray(cfg, s_inner, s_tri):
    """SURVEY.md §8(d): ray in + hit out + 2 packed nodes per inner step + one PrecomputedTri per test."""
    if cfg["dtype"] == "f64":
        return 64 + 32 + 128 * s_inner + 96 * s_tri
    return 32 + (4 if cfg["any_hit"] else 16) + 64 * s_inner + 48 * s_tri


def dump_outputs(out_dir, hits, hit_dtype):
    """Writes the hit records the timed path returned (all ranks' rays, in global ray order) as float arrays, so that
    two builds run with the same arguments can be compared output for output: prim_id (float64; exact for every id, a
    miss is the all-ones id), t, u, v (the config's precision) and ray_index (float64, the ray each record belongs to).
    Batches larger than DUMP_MAX_RAYS are represented by a fixed, seeded sample of DUMP_MAX_RAYS rays."""
    rec = hits.cpu().numpy().view(hit_dtype).reshape(-1)
    n = rec.shape[0]
    index = np.arange(n) if n <= DUMP_MAX_RAYS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_RAYS, replace=False))
    rec = rec[index]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("prim_id", rec["prim_id"].astype(np.float64)), ("t", rec["t"]), ("u", rec["u"]), ("v", rec["v"]),
                    ("ray_index", index.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU path on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_arm(cfg, kind, name, steps, warmup):
    """Times DefaultBuilder (Quality::High, the library default) and Bvh::intersect with every usable host
    thread on the rays of rank 0 (c4: every 10th image row).  Per-step times -> MEDIAN.  Only this function
    (and tests/, smoke()) touches oracle/."""
    from oracle.pyoracle import ANY_HIT, TIE_LOWEST_ID, Oracle, Ref, ref_available
    DYNAMIC = 1 << 8             # ref_driver.cpp kDynamic: workers claim 4096-ray blocks (no static n/threads split)
    tris = make_tris(cfg, kind)
    stride = C4_CPU_ROW_STRIDE if name == "c4" else 1
    rays = make_rays(cfg, kind, tris, row_stride=stride)
    flags = TIE_LOWEST_ID | (ANY_HIT if cfg["any_hit"] else 0)
    cpus = usable_cpus()
    what = "all rays of one rank's batch" if stride == 1 else f"every {stride}th row of the {cfg['img']}x{cfg['img']} camera"
    sample = f"{rays.shape[0]} rays ({what}), {tris.shape[0]} triangles, median of {steps} steps"
    if ref_available():
        ref = Ref()
        threads = cpus["usable"]
        cores = ref.thread_count(threads)
        bb, cc = ref.tri_bboxes_centers(tris)
        t0 = time.perf_counter()
        tree = ref.build(bb, cc, quality="high", threads=threads)
        build_s = time.perf_counter() - t0
        build_low_s = ref.time_build(bb, cc, quality="low", threads=threads)
        ref.set_triangles(tree, tris)
        times = []
        for i in range(warmup + steps):
            ref.trace(tree, rays, flags=flags | DYNAMIC, threads=threads, outputs=False)
            if i >= warmup:
                times.append(ref.last_trace_seconds)
        kind_ = "reference"
        ref.trace(tree, rays, flags=flags, threads=threads, outputs=False)       # the executor's static split, for the record
        static_mrays = rays.shape[0] / ref.last_trace_seconds / 1e6
        ref.trace(tree, rays[:200000], flags=flags, threads=-1, outputs=False)
        single = 200000 / ref.last_trace_seconds / 1e6
    else:
        orc = Oracle()
        cores = 1
        bb, cc = orc.tri_bboxes_centers(tris)
        t0 = time.perf_counter()
        tree = orc.build(bb, cc, quality="low")
        build_s = build_low_s = time.perf_counter() - t0
        orc.set_triangles(tree, tris)
        rays = rays[:: 16]
        sample = f"{rays.shape[0]} rays (every 16th ray; scalar port), {tris.shape[0]} triangles, median of {steps} steps"
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            orc.trace(tree, rays, flags=flags)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        kind_ = "port"
        single = static_mrays = rays.shape[0] / np.median(times) / 1e6
    med = float(np.median(times))
    return {"value": rays.shape[0] / med / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind_, "sample": sample,
            "ms_per_step": med * 1e3, "spread": {"min_ms": float(np.min(times)) * 1e3, "max_ms": float(np.max(times)) * 1e3},
            "schedule": "reference ThreadPool + ParallelExecutor, workers claim 4096-ray blocks",
            "static_split_mrays": static_mrays, "single_thread_mrays": single, "cpus": cpus,
            "build_high_mtris": tris.shape[0] / build_s / 1e6, "build_low_mtris": tris.shape[0] / build_low_s / 1e6}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    kind, name = args.mesh, args.config
    cfg = CONFIGS[name]
    workload = workload_text(cfg, kind, name)
    metric = cfg["metric"]

    if args.impl == "reference":
        if rank != 0:
            return
        res = cpu_arm(cfg, kind, name, args.steps, args.warmup)
        line = {"impl": "reference", "metric": metric, "value": res["value"], "unit": "Mrays/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
                "config": {"workload": workload, "bvh": "reference DefaultBuilder Quality::High", "sample": res["sample"],
                           "schedule": res["schedule"], "cpus": res["cpus"], "spread": res["spread"],
                           "static_split_mrays": res["static_split_mrays"], "single_thread_mrays": res["single_thread_mrays"]},
                "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "build": {"high_mtris_per_s": res["build_high_mtris"], "low_mtris_per_s": res["build_low_mtris"]},
                "e2e": {"value": res["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    numa = None
    if world > 1 and not args.no_numa:
        numa = bind_to_gpu_numa_node(local_rank)          # before torch allocates pinned memory

    import torch
    import torch.distributed as dist
    import bvh_b200.api as api
    from bvh_b200.multi_gpu import ShardedTracer

    if not torch.cuda.is_available() or api.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    api.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    stream = torch.cuda.Stream(device=device)
    torch.cuda.set_stream(stream)                 # everything below runs on this (non-default) stream,
    api.set_stream(stream.cuda_stream)            # library kernels included: CUDA events see them

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(values):
        t = torch.tensor(values, dtype=torch.float64, device=device).reshape(-1)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().tolist()

    # ---- inputs -----------------------------------------------------------------------------------
    dt = np_dtype(cfg)
    tdt = torch.float32 if dt == np.float32 else torch.float64
    sfx = "3f" if dt == np.float32 else "3d"
    ray_bytes, hit_bytes = (32, 16) if dt == np.float32 else (64, 32)
    hit_words = hit_bytes // 4
    hit_dtype = api.HIT3F if dt == np.float32 else api.HIT3D
    L = api.lib()
    tris_np = make_tris(cfg, kind)
    n_tris = tris_np.shape[0]
    verts = torch.from_numpy(tris_np).to(device)
    rays_np = make_rays(cfg, kind, tris_np, rank, world)
    n_rays = rays_np.shape[0]
    rays_pinned = torch.from_numpy(rays_np).pin_memory()
    rays = rays_pinned.to(device, non_blocking=True)
    torch.cuda.synchronize()
    total_rays = world * n_rays
    peak_gbs, peak_src = hbm_peak()
    base_flags = api.ANY_HIT if cfg["any_hit"] else 0
    kflag = {"auto": 0, "persistent": api.KERNEL_NO_TMA, "tma": api.KERNEL_TMA, "wide": api.KERNEL_WIDE,
             "simple": api.KERNEL_SIMPLE}[args.kernel]
    if args.sort_rays:
        kflag |= api.SORT_RAYS

    # ---- build: K timed LBVH builds from device-resident vertices ----------------------------------
    def build():
        return api.Bvh.build_triangles(verts.data_ptr(), count=n_tris, dtype=dt, flags=api.DEVICE_POINTERS, quality=args.quality)

    build_steps = args.steps if n_tris <= 2_000_000 else max(3, args.steps // 5)
    for _ in range(args.warmup):
        build().destroy()
    barrier()
    bev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(build_steps)]
    for s, e in bev:
        s.record()
        build().destroy()
        e.record()
    barrier()
    build_ms = float(np.median(max_over_ranks([s.elapsed_time(e) for s, e in bev])))
    bvh = build()
    props = bvh.properties()
    t0 = time.perf_counter()
    for _ in range(3):
        api.Bvh.build_triangles(tris_np, quality=args.quality).destroy()
    build_e2e_ms = (time.perf_counter() - t0) / 3 * 1e3
    morton_bits = int(props.get("morton_bits", 30))
    build_bytes = 300.0 if morton_bits <= 32 else 440.0        # SURVEY.md §8(d): bytes per triangle of the LBVH pipeline
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    build_info = {"value": n_tris / build_ms / 1e3, "unit": "Mtris/s", "ms": build_ms, "steps": build_steps, "scope": "per GPU (BVH replicated)",
                  "e2e_ms_host_vertices": build_e2e_ms, "depth": bvh.depth, "morton_bits": morton_bits,
                  "quality": args.quality or "high (library default)", "pipeline": props.get("pipeline"),
                  "roofline": {"bound": "hbm", "achieved": build_bytes * n_tris / (build_ms * 1e-3) / 1e9, "peak": peak_gbs,
                               "unit": "GB/s", "frac": build_bytes * n_tris / (build_ms * 1e-3) / 1e9 / peak_gbs,
                               "traffic": traffic_db.get(f"build_{kind}_{n_tris}"), "bytes_per_tri": build_bytes}}

    # ---- algorithmic bytes of the traversal, measured on the tree actually traversed, over the WHOLE timed batch
    st = torch.empty((n_rays, 3), dtype=torch.int32, device=device)
    scratch_hits = torch.empty((n_rays, hit_words), dtype=torch.int32, device=device)
    if getattr(L, f"bvh{sfx}_intersect_rays_stats")(bvh.handle, rays.data_ptr(), n_rays, scratch_hits.data_ptr(),
                                                    st.data_ptr(), api.DEVICE_POINTERS | base_flags):
        raise SystemExit(api.last_error())
    torch.cuda.synchronize()
    s_inner, s_leaves, s_tri = (float(x) for x in st.sum(dim=0, dtype=torch.float64).div(n_rays).tolist())
    if dt == np.float32:
        hit_frac = float((scratch_hits[:, 0] != -1).double().mean().item())
    else:
        hit_frac = float((scratch_hits.view(torch.int64)[:, 0] != -1).double().mean().item())
    bpr = bytes_per_ray(cfg, s_inner, s_tri)
    del st, scratch_hits

    # ---- traversal: W warm-up + K timed steps -------------------------------------------------------
    trace_fn = getattr(L, f"bvh{sfx}_intersect_rays")

    def trace(b, e, out):
        if trace_fn(bvh.handle, rays.data_ptr() + ray_bytes * b, e - b, out.data_ptr(), api.DEVICE_POINTERS | base_flags | kflag):
            raise SystemExit(api.last_error())

    tracer, gather_desc = None, None
    # auto: two ranks one multimem store per record (2-GPU run: 0.995 of perfect scaling, per-record peer stores 0.954, staged
    # 0.90); up to 4 ranks one peer store per record and rank (each costs ~1-2 % of the kernel: scripts/gather_probe.py); beyond
    # that warp-staged bulk copies (a fixed ~6 %, independent of the number of ranks) — ONE copy per 32 records to the multicast
    # address when the fabric has one (8 ranks: 0.881), else one copy per rank (0.836); NCCL (below) if none works
    candidates = gather_candidates(world, args.gather)
    for mode in candidates:
        try:
            from bvh_b200.multi_gpu import FusedGatherTracer
            api.set_option("gather_staging", 0 if mode in ("direct", "multicast") else 1)
            cand = FusedGatherTracer(bvh, rays, hit_words, flags=api.DEVICE_POINTERS | base_flags | kflag,
                                     mode="multicast" if mode.startswith("multicast") else "peer")
            how = ("one multimem.st per record through the NVSwitch multicast address" if mode == "multicast" else
                   "each warp stages the records of 32 consecutive rays in shared memory and sends the 512-byte block with ONE cp.async.bulk "
                   "to the NVSwitch multicast address" if mode == "multicast_staged" else
                   "one 16-byte NVLink peer store per record and rank" if mode == "direct" else
                   "each warp stages the records of 32 consecutive rays in shared memory and sends the 512-byte block to every rank "
                   "with one cp.async.bulk (shared -> peer global over NVLink)")
            # self-check before anything is timed: every rank must hold, for every shard, exactly the records its owner
            # gets from a plain (ungathered) launch
            truth = torch.empty((n_rays, hit_words), dtype=torch.int32, device=device)
            trace(0, n_rays, truth)
            cand.step()
            cand.check()
            torch.cuda.synchronize()
            got = cand.global_hits().view(world, n_rays, hit_words).to(torch.int64).sum(dim=(1, 2))
            owners = torch.empty(world, dtype=torch.int64, device=device)
            dist.all_gather_into_tensor(owners, truth.to(torch.int64).sum().reshape(1))
            good = torch.tensor([1 if torch.equal(got, owners) else 0], device=device)
            dist.all_reduce(good, op=dist.ReduceOp.MIN)
            del truth
            if not bool(good.item()):
                raise RuntimeError(f"fused gather ({mode}) delivered records that differ from the owners' plain launches")
            tracer = cand
            gather_desc = (f"fused in the traversal kernel into all {world} ranks' symmetric-memory buffers (double-buffered): {how}; "
                           "one symmetric-memory barrier per step")
            break
        except Exception as exc:
            if args.gather != "auto":
                raise
            if rank == 0:
                print(f"[bench] fused gather mode {mode} unavailable ({type(exc).__name__}: {exc})", file=sys.stderr)
    if tracer is None:
        tracer = ShardedTracer(n_rays, hit_words, torch.int32, device, trace, chunks=args.chunks if world > 1 else 1)
        if world > 1:
            gather_desc = f"NCCL all_gather_into_tensor of hit records, {args.chunks} chunks overlapped with traversal"
    for _ in range(max(3, args.warmup)):
        tracer.step()
    # Everything that can take host time (NVML initialisation of the clock sampler, event creation, a garbage collection)
    # happens BEFORE the barrier that opens the timed region: a rank that enters the region late makes every other rank
    # wait at the first step's symmetric-memory barrier, and that wait is inside their timed window (one 87 ms step in
    # a 20-step run halves the reported value: profiles/r02_n2_*).
    sampler = ClockSampler(local_rank)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    import gc
    gc.collect()
    gc.disable()
    barrier()
    e0.record()
    for k in range(args.steps):
        starts[k].record()
        tracer.step()
        ends[k].record()
    e1.record()
    barrier()
    gc.enable()
    if hasattr(tracer, "check"):
        tracer.check()                           # a fired kernel watchdog means stale records: fail, do not report
    clocks = sampler.summary()
    total_ms = max_over_ranks([e0.elapsed_time(e1)])[0]
    ms_per_step = total_ms / args.steps
    step_ms = max_over_ranks([s.elapsed_time(e) for s, e in zip(starts, ends)])     # per step, max over ranks
    kernel_ms = float(np.median(step_ms))
    value = total_rays / ms_per_step / 1e3                     # Mrays/s, whole job
    kernel_name = bvh.properties().get("last_kernel", "trace_persistent_kernel")

    hits_np = tracer.local.cpu().numpy().view(hit_dtype).reshape(-1)
    checksum = int(hits_np["prim_id"].astype(np.uint64).sum() & np.uint64(0xFFFFFFFFFFFFFFFF))
    if world > 1:
        g = tracer.global_hits()
        assert g.shape[0] == total_rays
        assert torch.equal(g[rank * n_rays:(rank + 1) * n_rays], tracer.local), "gathered hits do not match the local shard"
        # every rank must hold every other rank's shard: compare per-shard checksums across ranks
        sums = g.view(world, n_rays, hit_words)[:, :, 0].to(torch.int64).sum(dim=1)
        ref_sums = sums.clone()
        dist.broadcast(ref_sums, src=0)
        assert torch.equal(sums, ref_sums), "ranks disagree on the gathered hit records"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tracer.global_hits(), hit_dtype)

    # ---- e2e through the C ABI with pinned host buffers ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        hits_pinned = torch.empty((n_rays, hit_words), dtype=torch.int32).pin_memory()

        def call():
            if trace_fn(bvh.handle, rays_pinned.data_ptr(), n_rays, hits_pinned.data_ptr(), base_flags | kflag):
                raise SystemExit(api.last_error())
        for _ in range(2):
            call()
        barrier()
        e2e_steps = args.steps if n_rays <= 20_000_000 else max(3, args.steps // 5)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            call()
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks([(time.perf_counter() - t0) / e2e_steps * 1e3])[0]
        assert np.array_equal(hits_pinned.numpy().view(hit_dtype).reshape(-1), hits_np), "e2e hits differ from device-resident hits"
        e2e = {"value": total_rays / e2e_ms / 1e3, "unit": "Mrays/s", "ms_per_step": e2e_ms, "steps": e2e_steps,
               "h2d_bytes_per_step": int(n_rays * ray_bytes), "d2h_bytes_per_step": int(n_rays * hit_bytes),
               "api": f"bvh{sfx}_intersect_rays(host rays, host hits) with pinned buffers", "numa": numa}

    # ---- CPU baseline beside it (rank 0, N = 1 only) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = cpu_arm(cfg, kind, name, 5, 2)
        cpu = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cpu.update(single_thread_mrays=res["single_thread_mrays"], static_split_mrays=res["static_split_mrays"],
                   build_high_mtris=res["build_high_mtris"], build_low_mtris=res["build_low_mtris"], spread=res["spread"])

    if rank == 0:
        achieved = bpr * n_rays / (kernel_ms * 1e-3) / 1e9       # one launch = one rank's shard
        line = {
            "metric": metric, "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
            "config": {"workload": workload, "bvh": f"{props.get('pipeline', 'LBVH')} built on the GPU, replicated per rank",
                       "kernel": kernel_name, "tie_break": "lowest original id (canonical)",
                       "ray_order": "Morton order of the origins (device radix sort inside every step)" if args.sort_rays else "as given",
                       "l2": f"inputs larger than L2: {n_rays * ray_bytes / 1e6:.0f} MB of rays + {n_rays * hit_bytes / 1e6:.0f} MB of hits streamed per step, no flush needed",
                       "hit_fraction": hit_frac, "inner_steps_per_ray": s_inner, "leaves_per_ray": s_leaves, "tri_tests_per_ray": s_tri,
                       "stats_rays": n_rays, "gather": gather_desc, "hits_checksum": checksum,
                       "step_ms": {"median": kernel_ms, "max": float(np.max(step_ms)), "min": float(np.min(step_ms)),
                                   "slow_steps": [[int(i), float(t)] for i, t in enumerate(step_ms) if t > 1.5 * kernel_ms]}},
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak_gbs,
                         "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "traffic": traffic_db.get(f"trace_{name}_{kind}"),
                         "bytes_per_ray": bpr, "launch_ms": kernel_ms,
                         "note": "algorithmic bytes over time; the tree is L2-resident, so frac can exceed 1 (traffic = DRAM bytes per launch, ncu)"},
            "build": build_info,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": args.steps * len(tracer.bounds),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
