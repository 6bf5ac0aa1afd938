#!/usr/bin/env python3
"""bench.py — BASELINE.json's metric (ICP correspondences/s, ms/iteration, HBM GB/s of the search against the roofline).

Default workload (config.workload = "cfg3_10M_point_to_plane", BASELINE.json configs[2], SURVEY.md §8d — the 10 M-point
configuration the metric is quoted on):
  target : 10 000 000 points, (x,y) ~ U[0,10)^2, z = 0.5 sin(x) cos(0.7 y) + N(0, 0.002^2), seed 7
  source : the same surface re-sampled (seed 8 + rank), rotated 2 deg about z, t = (0.02, 0.01, -0.01)
  target normals: NormalEstimation k = 16, viewpoint (5,5,10)  (set-up, timed separately, not part of a step)
  ICP    : IterativeClosestPointWithNormals (non-symmetric => TransformationEstimationPointToPlaneLLS),
           max correspondence distance 0.05, k = 1
A STEP is one Registration::align() of ICP_ITERS iterations (10 = PCL's default max_iterations_, registration.h:566)
over the whole source cloud: source upload -> Hilbert ordering of the queries -> ICP_ITERS x (transform + exact 1-NN +
gate + normal-equation accumulation + solve) -> output cloud.  The target index is built once before the timed region,
exactly as pcl::Registration keeps its tree across align() calls (registration.hpp:84-87).
  value : correspondences/s with source, target index and output resident in HBM (device pointers through the same
          C-ABI calls pclb200_icp_set_source / _iterate / _get_cloud the C++ facade's align() makes)
  e2e   : the same calls with HOST buffers (pinned records): H2D of the source and D2H of the aligned cloud inside the
          timed region
Other workloads (--workload, SURVEY.md §8d table; the driver's default run is cfg3):
  cfg4 : 50 M-point scene of 40 planar patches in [0,20)^3 + N(0,0.005^2); source re-sampled, rotated 1 deg about a
         random axis, |t| = 0.02; point-to-point (TransformationEstimationSVD), gate 0.05; intended for 4 GPUs
  cfg5 : 200 M-ray spinning-LiDAR sweep (64 beams) of a 200 m x 30 m street canyon (ground, two facades, end walls),
         range noise N(0,0.02^2); second sweep after ego-motion (yaw 1.5 deg, t = (0.5,0.1,0)); both clouds through
         VoxelGrid leaf 0.1 (the finest leaf below the INT32 guard, voxel_grid.hpp:620-629), then ICP SVD with exactly 30
         iterations (all epsilons 0); intended for 8 GPUs
Scaling (--scaling):
  weak   : every rank holds a replica of the target index and its OWN source cloud of the full size (default)
  strong : ONE source, cut into spatial tiles (chunks of 65 536 Morton-consecutive points dealt round-robin to the ranks;
           --shard contiguous = one Morton range per rank), so per-GPU work shrinks with N.  The 40 fp64 accumulators are exchanged once per iteration over NVLink (fused into the
           accumulate kernel's last block; NCCL bootstraps the peer mappings).
--impl reference times the CPU restatement of PCL's own path (oracle/; the reference itself cannot be compiled in this
image: no Eigen/Boost/FLANN) on the box's host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ICP_ITERS = 10
MAX_CORR_DIST = 0.05
N_DEFAULT = 10_000_000
_JSON_OUT = sys.stdout
METRIC = "icp_correspondences_per_sec"
UNIT = "correspondences/s"


# -----------------------------------------------------------------------------------------------------------------
# cfg3: Gaussian surface (records = pcl::PointNormal, 12 floats)
# -----------------------------------------------------------------------------------------------------------------
def surface(n, seed):
    r = np.random.default_rng(seed)
    xy = r.random((n, 2)) * 10.0
    z = 0.5 * np.sin(xy[:, 0]) * np.cos(0.7 * xy[:, 1]) + r.normal(0.0, 0.002, n)
    return xy[:, 0], xy[:, 1], z


def make_target(n):
    x, y, z = surface(n, 7)
    t = np.zeros((n, 12), dtype=np.float32)  # pcl::PointNormal records
    t[:, 0], t[:, 1], t[:, 2], t[:, 3] = x, y, z, 1.0
    return t


def make_source(n, rank):
    x, y, z = surface(n, 8 + rank)
    a = np.deg2rad(2.0)
    c, s = np.cos(a), np.sin(a)
    out = np.zeros((n, 12), dtype=np.float32)
    out[:, 0] = c * x - s * y + 0.02
    out[:, 1] = s * x + c * y + 0.01
    out[:, 2] = z - 0.01
    out[:, 3] = 1.0
    return out


def analytic_normals(t, vp=(5.0, 5.0, 10.0)):
    """Normals of z = 0.5 sin x cos 0.7y (used by the REFERENCE arm only: it may not call our normals kernel)."""
    x, y = t[:, 0].astype(np.float64), t[:, 1].astype(np.float64)
    n = np.stack([-0.5 * np.cos(x) * np.cos(0.7 * y), 0.35 * np.sin(x) * np.sin(0.7 * y), np.ones_like(x)], 1)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    flip = ((np.asarray(vp) - t[:, :3]) * n).sum(1) < 0
    n[flip] *= -1
    return n.astype(np.float32)


# -----------------------------------------------------------------------------------------------------------------
# cfg4: scene of planar patches (records = pcl::PointXYZ, 4 floats)
# -----------------------------------------------------------------------------------------------------------------
def _scene_patches():
    r = np.random.default_rng(11)
    patches = []
    for _ in range(40):
        c = r.uniform(3.0, 17.0, 3)
        u = r.normal(size=3)
        u /= np.linalg.norm(u)
        w = r.normal(size=3)
        v = np.cross(u, w)
        v /= np.linalg.norm(v)
        patches.append((c, u * r.uniform(2.0, 6.0), v * r.uniform(2.0, 6.0)))
    return patches


def scene_points(n, seed):
    patches = _scene_patches()
    r = np.random.default_rng(seed)
    area = np.array([np.linalg.norm(np.cross(u, v)) for (_, u, v) in patches])
    counts = np.floor(n * area / area.sum()).astype(np.int64)
    counts[0] += n - counts.sum()
    out = np.empty((n, 4), dtype=np.float32)
    k = 0
    for (c, u, v), m in zip(patches, counts):
        ab = r.uniform(-0.5, 0.5, (m, 2)).astype(np.float32)
        p = c.astype(np.float32) + ab[:, :1] * u.astype(np.float32) + ab[:, 1:] * v.astype(np.float32)
        p += r.normal(0.0, 0.005, (m, 3)).astype(np.float32)
        out[k:k + m, :3] = np.clip(p, 0.0, np.float32(19.999))
        k += m
    out[:, 3] = 1.0
    return out


def scene_source(n, seed):
    p = scene_points(n, seed)
    r = np.random.default_rng(12)
    ax = r.normal(size=3)
    ax /= np.linalg.norm(ax)
    a = np.deg2rad(1.0)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * (K @ K)
    t = r.normal(size=3)
    t *= 0.02 / np.linalg.norm(t)
    c = np.array([10.0, 10.0, 10.0])
    q = (p[:, :3].astype(np.float64) - c) @ R.T + c + t
    p[:, :3] = q.astype(np.float32)
    return p


# -----------------------------------------------------------------------------------------------------------------
# cfg5: spinning-LiDAR sweep of a street canyon (records = pcl::PointXYZ)
# -----------------------------------------------------------------------------------------------------------------
def lidar_sweep(n_rays, seed, yaw_deg=0.0, tx=0.0, ty=0.0, chunk=25_000_000, device=None):
    """n_rays rays of a 64-beam spinning sensor at world (tx, ty, 2) with heading yaw; returns the hits in the SENSOR
    frame (x forward) as an (m, 4) float32 numpy array.  Scene: ground z = 0, facades y = +-15 (20 m high), end walls
    x = +-100; max range 120 m.  Generated with torch (on `device` when given: 200 M rays take seconds on the GPU and
    minutes in numpy); the stream depends on the device type, the distribution does not."""
    import torch
    dev = torch.device(device if device is not None else "cpu")
    g = torch.Generator(device=dev)
    g.manual_seed(int(seed))
    elev = torch.deg2rad(torch.linspace(-25.0, 15.0, 64, device=dev))
    yaw = float(np.deg2rad(yaw_deg))
    c, sn = float(np.cos(yaw)), float(np.sin(yaw))
    inf = float("inf")
    out = []
    for s in range(0, n_rays, chunk):
        m = min(chunk, n_rays - s)
        az = torch.rand(m, generator=g, device=dev) * (2 * np.pi) + yaw
        el = elev[torch.randint(0, 64, (m,), generator=g, device=dev)]
        ce = torch.cos(el)
        dx, dy, dz = ce * torch.cos(az), ce * torch.sin(az), torch.sin(el)  # world direction
        del az, el, ce
        t = torch.where(dz < 0, -2.0 / dz, torch.full_like(dz, inf))
        for d_ax, o_ax, planes in ((dy, ty, (-15.0, 15.0)), (dx, tx, (-100.0, 100.0))):
            for pl in planes:
                tt = (pl - o_ax) / d_ax
                z = 2.0 + tt * dz
                ok = (tt > 0) & (z >= 0) & (z <= 20.0)
                t = torch.minimum(t, torch.where(ok, tt, torch.full_like(tt, inf)))
        ok = torch.isfinite(t) & (t < 120.0)
        t = t[ok]
        t = t + torch.randn(t.shape[0], generator=g, device=dev) * 0.02
        hx, hy, hz = t * dx[ok], t * dy[ok], 2.0 + t * dz[ok]   # hit relative to the sensor's ground position
        p = torch.ones((t.shape[0], 4), dtype=torch.float32, device=dev)
        p[:, 0] = c * hx + sn * hy   # world -> sensor frame
        p[:, 1] = -sn * hx + c * hy
        p[:, 2] = hz
        out.append(p.cpu())
        del dx, dy, dz, t, ok, hx, hy, hz, p
    return torch.cat(out, 0).numpy()


WORKLOADS = {
    "cfg3": dict(name="cfg3_10M_point_to_plane", n=N_DEFAULT, iters=ICP_ITERS, gate=MAX_CORR_DIST, width=12,
                 estimator="point_to_plane_lls", normals_k=16, voxel_leaf=None),
    "cfg4": dict(name="cfg4_50M_scene_gate_0.05", n=50_000_000, iters=ICP_ITERS, gate=0.05, width=4,
                 estimator="svd", normals_k=0, voxel_leaf=None),
    "cfg5": dict(name="cfg5_200M_lidar_voxelgrid_30iters", n=200_000_000, iters=30, gate=1.0, width=4,
                 estimator="svd", normals_k=0, voxel_leaf=0.1),
}


def gen_clouds(wl, n, rank, strong, device=None):
    """(target records, full source records) as numpy arrays; under strong scaling every rank generates the same source."""
    src_rank = 0 if strong else rank
    if wl == "cfg3":
        return make_target(n), make_source(n, src_rank)
    if wl == "cfg4":
        return scene_points(n, 11), scene_source(n, 13 + src_rank)
    return lidar_sweep(n, 21, device=device), lidar_sweep(n, 22 + src_rank, yaw_deg=1.5, tx=0.5, ty=0.1, device=device)


def morton_order(xyz):
    """argsort by a 30-bit Morton code of the cloud's own bounding box (host side, set-up only)."""
    lo = xyz.min(0)
    ext = float((xyz.max(0) - lo).max()) or 1.0
    q = np.minimum(((xyz - lo) * (1023.999 / ext)).astype(np.uint32), 1023)

    def spread(v):
        v = v.astype(np.uint64)
        v = (v | (v << 16)) & np.uint64(0x030000FF)
        v = (v | (v << 8)) & np.uint64(0x0300F00F)
        v = (v | (v << 4)) & np.uint64(0x030C30C3)
        v = (v | (v << 2)) & np.uint64(0x09249249)
        return v
    key = spread(q[:, 0]) | (spread(q[:, 1]) << np.uint64(1)) | (spread(q[:, 2]) << np.uint64(2))
    return np.argsort(key, kind="stable")


SHARD_CHUNK = 65536


def shard_strong(src, rank, world, mode="cyclic"):
    """rank r's share of the ONE source cloud, as spatial tiles: the cloud in Morton order is cut into chunks of
    SHARD_CHUNK consecutive points (compact patches) that are dealt round-robin to the ranks ("cyclic", default), or into
    `world` contiguous ranges ("contiguous").  Equal point counts either way; the cyclic deal also equalises the WORK —
    a rigid motion displaces one end of the cloud more than the other, walks there are longer, and with one contiguous
    range per rank the fastest rank waits in the per-iteration exchange (measured at N = 2: 17.5 ms per step, 6.3 ms
    of it spent waiting in the accumulate kernel, profiles/r2n_cfg3_strong_2gpu_contiguous.json)."""
    if world == 1:
        return src
    order = morton_order(src[:, :3])
    n = src.shape[0]
    if mode == "contiguous":
        lo, hi = (n * rank) // world, (n * (rank + 1)) // world
        mine = order[lo:hi]
    else:
        chunk = np.arange(n) // SHARD_CHUNK
        mine = order[(chunk % world) == rank]
    return np.ascontiguousarray(src[np.sort(mine)])


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML (in-process thread; the same
    counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints, B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index, period_s=0.05):
        self.gpu, self.period = gpu_index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.th = None
        self.err = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[0].isdigit() else self.gpu
            self.h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.nv = nv
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
        except Exception as e:  # noqa
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake_slowdown": 0x80}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, b in bits.items():
                    if r & b:
                        self.reasons.add(k)
            except Exception as e:  # noqa
                self.err = repr(e)
                break
            self.stop_flag.wait(self.period)

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "samples": len(self.sm), "reasons": sorted(self.reasons), "how": "NVML, 50 ms period, timed region only"}
        if self.err:
            out["error"] = self.err
        return out


def measured_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(kernel_key, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu capture
    (profiles/ncu_traffic.json, written from a `ncu --set full` run of this workload); None when no capture matches."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = t.get(kernel_key)
        if e and int(e.get("points", -1)) == int(n):
            return float(e["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def host_cores():
    return int(os.cpu_count() or 1)


# -----------------------------------------------------------------------------------------------------------------
# reference arm: the CPU restatement of PCL's path (oracle/), all host threads, bounded sample
# -----------------------------------------------------------------------------------------------------------------
def oracle_kw(W, cores, tree):
    return dict(max_iterations=W["iters"], max_correspondence_distance=W["gate"],
                estimator=1 if W["estimator"] == "point_to_plane_lls" else 0,
                with_normals_transform=W["estimator"] == "point_to_plane_lls",
                source_has_normals=W["estimator"] == "point_to_plane_lls", nthreads=cores, index=tree)


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import oracle
    W = WORKLOADS[args.workload]
    n = args.points or W["n"]
    cores = host_cores()
    tgt, src_full = gen_clouds(args.workload, n, 0, False)
    if args.workload == "cfg3":
        tgt[:, 4:7] = analytic_normals(tgt)
    if W["voxel_leaf"]:
        # the reference pipeline's front-end (VoxelGrid on both clouds), untimed here like the kd-tree build
        tgt = oracle.voxelgrid(tgt, [W["voxel_leaf"]] * 3)
        src_full = oracle.voxelgrid(src_full, [W["voxel_leaf"]] * 3)
    t0 = time.time()
    tree = oracle.Index(tgt)  # pcl::KdTreeFLANN::setInputCloud, kept across align() calls
    build_s = time.time() - t0
    kw = oracle_kw(W, cores, tree)
    # calibrate the sample so that (steps + warmup) aligns end within ~150 s
    probe = min(src_full.shape[0], 100_000)
    t0 = time.time()
    r = oracle.icp_align(src_full[:probe], tgt, want_cloud=True, **kw)
    rate = max(r["total_correspondences"], 1) / max(time.time() - t0, 1e-6)
    budget_s = 150.0 / max(args.steps + args.warmup, 1)
    sample = int(min(src_full.shape[0], max(probe, rate * budget_s / W["iters"])))
    src = np.ascontiguousarray(src_full[:sample])
    out = np.empty_like(src)
    for _ in range(args.warmup):
        oracle.icp_align(src, tgt, out=out, **kw)
    total, t0 = 0, time.time()
    for _ in range(args.steps):
        r = oracle.icp_align(src, tgt, out=out, **kw)
        total += r["total_correspondences"]
    dt = time.time() - t0
    val = total / dt
    sample_desc = (f"{sample} of {src_full.shape[0]} source points (first rows) x {W['iters']} iterations per step against "
                   f"the full {tgt.shape[0]}-point target; kd-tree build ({build_s:.1f} s, 1 thread) outside the timed "
                   "region" + ("; analytic target normals" if args.workload == "cfg3" else ""))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": W["name"], "points_target": int(tgt.shape[0]), "points_source_per_step": sample,
                       "icp_iterations_per_step": W["iters"], "max_correspondence_distance": W["gate"],
                       "estimator": W["estimator"], "k": 1},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample_desc},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


# -----------------------------------------------------------------------------------------------------------------
# our arm
# -----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import pcl_b200 as P
    rank, world, local = dist_env()
    W = WORKLOADS[args.workload]
    n = args.points or W["n"]
    strong = args.scaling == "strong"
    p2plane = W["estimator"] == "point_to_plane_lls"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    P.lib()
    ctx = P.Context(local)
    if world > 1:
        uid = [P.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    # ---- set-up (outside the timed region): clouds, target-side VoxelGrid, target index, normals -------------------------
    tgt, src_full = gen_clouds(args.workload, n, rank, strong, device=dev)
    setup_ms = {}
    ctx.profile(True)
    leaf = W["voxel_leaf"]
    grid_bounds = None
    if leaf:
        # cfg5.  Target: one VoxelGrid over the whole sweep (set-up, like the index build).  Source: the RAW sweep is cut
        # into spatial tiles along voxel columns of the WHOLE sweep's grid; every step each rank filters its tile on that
        # grid (pclb200_voxelgrid_tile: the tiles' voxels are exactly the voxels of one VoxelGrid over the whole sweep)
        # and aligns the result — the downsample front-end is part of the step and shards with the source.
        a = torch.from_numpy(tgt).to(dev)
        o = torch.empty_like(a)
        ctx.profile_reset()
        f = ctx.voxelgrid(a, [leaf] * 3, out=o)
        setup_ms["voxelgrid_target"] = ctx.profile_get("voxelgrid")[0]
        setup_ms["voxelgrid_target_points_in"] = int(a.shape[0])
        tgt = f.cpu().numpy().copy()
        del a, o, f
        torch.cuda.empty_cache()
        lo, hi = src_full[:, :3].min(0), src_full[:, :3].max(0)
        grid_bounds = np.concatenate([lo, hi]).astype(np.float32)
        if strong and world > 1:
            inv = np.float32(1.0) / np.float32(leaf)
            col = (np.floor(src_full[:, 0] * inv) - np.floor(lo[0] * inv)).astype(np.int64)
            cum = np.cumsum(np.bincount(col))
            cuts = [0] + [int(np.searchsorted(cum, cum[-1] * r / world)) + 1 for r in range(1, world)] + [int(col.max()) + 1]
            src_full = np.ascontiguousarray(src_full[(col >= cuts[rank]) & (col < cuts[rank + 1])])
            del col
    n_tgt = int(tgt.shape[0])
    n_src_total = int(src_full.shape[0]) * (1 if (strong and not leaf) else world)
    if leaf:
        src_np = src_full                                  # this rank's raw tile (strong) / own sweep (weak)
        if strong and world > 1:
            t = torch.tensor([float(src_np.shape[0])], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            n_src_total = int(t[0])
    else:
        src_np = shard_strong(src_full, rank, world, args.shard) if strong else src_full
    del src_full
    src_host = torch.from_numpy(src_np).pin_memory()
    ctx.profile_reset()
    tidx = P.Index(ctx, tgt)
    setup_ms["index_build"] = ctx.profile_get("index_build")[0]
    nrm_dev = None
    if p2plane:
        tgt_dev = torch.from_numpy(tgt).to(dev)
        nrm_dev = torch.empty((n_tgt, 4), dtype=torch.float32, device=dev)
        tidx.normals_knn(tgt_dev, W["normals_k"], viewpoint=(5.0, 5.0, 10.0), out=nrm_dev)
        setup_ms[f"normals_k{W['normals_k']}_first_call"] = ctx.profile_get("normals")[0]   # incl. first-use allocations
        ctx.profile_reset()
        tidx.normals_knn(tgt_dev, W["normals_k"], viewpoint=(5.0, 5.0, 10.0), out=nrm_dev)
        setup_ms[f"normals_k{W['normals_k']}"] = ctx.profile_get("normals")[0]
        del tgt_dev
    src_dev = src_host.to(dev)                    # value leg: records already resident in HBM
    vg_buf = None
    n_filtered = int(src_np.shape[0])
    if leaf:
        vg_buf = torch.empty_like(src_dev)
        n_filtered = int(ctx.voxelgrid_tile(src_dev, [leaf] * 3, grid_bounds, out=vg_buf).shape[0])
        out_host = torch.empty((n_filtered, src_host.shape[1]), dtype=torch.float32).pin_memory()
        out_dev = torch.empty((n_filtered, src_host.shape[1]), dtype=torch.float32, device=dev)
    else:
        out_host = torch.empty_like(src_host).pin_memory()
        out_dev = torch.empty_like(src_dev)
    params = P.default_params(max_iterations=W["iters"], max_correspondence_distance=W["gate"],
                              estimator=P.EST_POINT_TO_PLANE_LLS if p2plane else P.EST_SVD,
                              with_normals_transform=1 if p2plane else 0, mse_threshold_absolute=0.0,
                              transformation_epsilon=0.0)

    # One registration object for the whole run, like a pcl::IterativeClosestPoint[WithNormals] instance whose target
    # was set once (Registration::setInputTarget): the target index and its normals stay on the device across
    # align() calls (registration.hpp:84-87); every step is setInputSource + align(output).
    def make_aligner(cx, vg):
        obj = P.Icp(cx, params=params)
        obj.set_target(tidx, normals=nrm_dev)

        def align(src, out):
            if leaf:
                src = cx.voxelgrid_tile(src, [leaf] * 3, grid_bounds, out=vg)   # the step's downsample front-end
            if p2plane:
                obj.set_source(src, normals=P.Field(src, 4))
            else:
                obj.set_source(src)
            st = obj.iterate()
            if p2plane:
                obj.get_cloud(out, normals=P.Field(out, 4))
            else:
                obj.get_cloud(out)
            return st
        return align

    align = make_aligner(ctx, vg_buf)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(src, out, steps, warmup, sample_clocks):
        for _ in range(warmup):
            align(src, out)
        ctx.profile_reset()
        l0 = ctx.launches
        barrier()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total, iters = 0, 0
        st = None
        e0.record(stream)
        for _ in range(steps):
            st = align(src, out)
            total += st["total_correspondences"]
            iters += st["iterations"]
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if sampler else None
        ms = e0.elapsed_time(e1)
        if world > 1:
            tm = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm[0])
        # with the exchange inside every iteration each rank's stats already carry the GLOBAL pair counts
        return ms, float(total), ctx.launches - l0, clocks, iters, st

    # device-resident leg (value) --------------------------------------------------------------------------------
    ms_v, tot_v, launches, clocks, iters_v, last_v = timed(src_dev, out_dev, args.steps, args.warmup, not args.no_clocks)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_v, out_dev, p2plane)
    prof = {k: ctx.profile_get(k) for k in ("icp_search", "icp_accum", "allreduce", "query_sort", "solve", "transform_out",
                                            "voxelgrid")}
    # host-buffer leg (e2e) --------------------------------------------------------------------------------------
    ms_e1, tot_e1, _, _, _, _ = timed(src_host, out_host, args.steps, max(1, args.warmup // 2), False)
    ms_e, tot_e, depth = ms_e1, tot_e1, 1
    pipeline_error = None
    if world == 1 and not args.no_pipeline:
        try:
            # The same K steps with TWO aligns in flight, as a consumer registering a stream of scans double-buffers them: a
            # second registration object on its own context (= its own stream) and its own pinned buffers, one host thread
            # per object (the C-ABI calls release the GIL).  Every step still uploads its source and downloads its aligned
            # cloud inside the timed region; what overlaps is one step's PCIe copies with the other step's kernels.
            import threading
            ctx_b = P.Context(local)
            align_b = make_aligner(ctx_b, torch.empty_like(vg_buf) if vg_buf is not None else None)
            src_host_b = src_host.clone().pin_memory()
            out_host_b = torch.empty_like(out_host).pin_memory()
            lanes = [(align, src_host, out_host), (align_b, src_host_b, out_host_b)]
            for fn, a_src, a_out in lanes:
                for _ in range(2):
                    fn(a_src, a_out)
            share = [args.steps - args.steps // 2, args.steps // 2]
            res = [None, None]

            def run(k):
                fn, a_src, a_out = lanes[k]
                tot = 0.0
                try:
                    for _ in range(share[k]):
                        tot += fn(a_src, a_out)["total_correspondences"]
                    res[k] = tot
                except Exception as e:   # noqa: BLE001 — re-raised on the main thread
                    res[k] = e
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            th = [threading.Thread(target=run, args=(k,)) for k in range(2)]
            for t in th:
                t.start()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            e1.record(stream)
            torch.cuda.synchronize()
            for r_ in res:
                if isinstance(r_, Exception):
                    raise r_
            ms_e, tot_e, depth = e0.elapsed_time(e1), float(sum(res)), 2
        except Exception as e:   # noqa: BLE001 — the one-at-a-time figure stands, the reason is reported
            pipeline_error = repr(e)
            print(f"[bench] pipelined e2e leg failed, keeping the single-in-flight figure: {e!r}", file=sys.stderr)
            ms_e, tot_e, depth = ms_e1, tot_e1, 1
    value = tot_v / (ms_v * 1e-3)
    e2e = tot_e / (ms_e * 1e-3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (SURVEY.md §8(d)) ----------------------------------------------------------
    # k_search = in-place transform + exact seeded 1-NN + gate of one ICP iteration (>= 85 % of a step).
    # ALGORITHMIC bytes per correspondence (§8d): 16 (query read) + 24 * N_t / N_s (every target point, 16 B, and its
    # share of a 32-B node per 8-point leaf, read once under coherent queries) = 40 B at N_s = N_t.  The whole iteration
    # (k_search + k_accum_dmma) adds 16 * N_t / N_s for the target normals of the point-to-plane objective = 56 B; it is
    # reported as `iteration`.  The implementation moves more than that (the in-place fp32 re-transform of the source
    # that reproduces icp.hpp:220 bit for bit, the 8-B match = next iteration's seed, leaf padding, 64-B nodes, the cell
    # table): `implementation_bytes_per_correspondence`; the DRAM bytes ncu measured per launch are `traffic`.
    st_idx = tidx.stats
    n_local = n_filtered
    ratio = n_tgt / float(n_local)
    alg_search = 16.0 + 24.0 * ratio
    alg_iter = alg_search + (16.0 * ratio if p2plane else 0.0)
    impl_bytes = (16 + 16 + 8 + 8 + (st_idx["leaves"] * st_idx["leaf_size"] * 16 + st_idx["nodes"] * 64) / float(n_local))
    peak, peak_src = measured_peak_gbs()
    iter_ms, iter_n = prof["icp_search"]
    acc_ms, acc_n = prof["icp_accum"]
    avg_search_s = (iter_ms / max(iter_n, 1)) * 1e-3
    avg_iter_s = avg_search_s + (acc_ms / max(acc_n, 1)) * 1e-3
    achieved = alg_search * n_local / avg_search_s / 1e9 if avg_search_s > 0 else 0.0
    ach_iter = alg_iter * n_local / avg_iter_s / 1e9 if avg_iter_s > 0 else 0.0
    roofline = {"bound": "hbm",
                "kernel": "k_search (in-place transform + exact seeded 1-NN started at the candidate ball + gate)",
                "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_nominal_8000_GBs": achieved / 8000.0,  # SURVEY.md §8(d): report both denominators
                "traffic": ncu_traffic("k_search_" + args.workload, n),
                "algorithmic_bytes_per_launch": alg_search * n_local, "avg_launch_ms": avg_search_s * 1e3,
                "launches_timed": iter_n, "algorithmic_bytes_per_correspondence": alg_search,
                "implementation_bytes_per_correspondence": impl_bytes,
                "iteration": {"kernels": "k_search + k_accum_dmma", "algorithmic_bytes_per_correspondence": alg_iter,
                              "avg_ms": avg_iter_s * 1e3, "achieved": ach_iter, "frac": ach_iter / peak,
                              "accum_kernel_ms": acc_ms / max(acc_n, 1),
                              "accum_kernel_GBs_of_its_56B": ((8 + 16 + 16 + (16 if p2plane else 0)) * n_local /
                                                             max(acc_ms / max(acc_n, 1) * 1e-3, 1e-12) / 1e9)},
                "index": st_idx,
                "note": "the walk is latency/issue bound, not HBM bound (SURVEY.md §7 hard part ii, DESIGN.md §3); frac "
                        "is the §8(d) algorithmic figure over the measured copy peak"}

    # CPU baseline (oracle port) on a bounded sample: one align(), sample sized for ~15 s, all host threads
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        import oracle
        cores = host_cores()
        tgt_n = tgt.copy()
        if p2plane:
            tgt_n[:, 4:8] = nrm_dev.cpu().numpy()
        t0 = time.time()
        tree = oracle.Index(tgt_n)
        build_s = time.time() - t0
        kw = oracle_kw(W, cores, tree)
        if leaf:   # the CPU arm aligns the filtered cloud too (its own VoxelGrid outside the sample timing)
            src_np = oracle.voxelgrid(src_np, [leaf] * 3)
        probe = min(n_local, 100_000)
        t0 = time.time()
        r = oracle.icp_align(src_np[:probe], tgt_n, **kw)
        rate = max(r["total_correspondences"], 1) / max(time.time() - t0, 1e-6)
        sample = int(min(n_local, max(probe, rate * 15.0 / W["iters"])))
        t0 = time.time()
        r = oracle.icp_align(np.ascontiguousarray(src_np[:sample]), tgt_n, want_cloud=True, **kw)
        dt = time.time() - t0
        cpu = {"value": r["total_correspondences"] / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{sample} of {n_local} source points x {W['iters']} iterations (one align) against the full "
                         f"{n_tgt}-point target" + (", GPU-computed normals" if p2plane else "") +
                         f"; kd-tree build {build_s:.1f} s excluded"}

    rec_bytes = int(src_host.numel() * 4)
    out_bytes = int(out_host.numel() * 4)
    steps = max(args.steps, 1)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_v / steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": W["name"], "points_target": n_tgt, "points_source_total": n_src_total,
                       "points_source_per_gpu": int(src_np.shape[0]), "points_aligned_per_gpu": n_local,
                       "icp_iterations_per_step": W["iters"],
                       "max_correspondence_distance": W["gate"], "estimator": W["estimator"], "k": 1,
                       "normals_k": W["normals_k"], "voxel_leaf": W["voxel_leaf"],
                       "l2_policy": "inputs larger than L2 (target points + nodes + normals + source >> 126 MB)",
                       "parallelism": (f"source sharded x{world} ({'Morton tiles of one cloud, ' + args.shard if strong else 'one cloud per rank'}), "
                                       "target replicated, 40-double exchange per iteration fused into the accumulate kernel")},
            "ms_per_iter": ms_v / max(iters_v, 1),
            "breakdown_ms_per_step": {"icp_iteration_kernel": prof["icp_search"][0] / steps,
                                      "icp_accum_kernel": prof["icp_accum"][0] / steps,
                                      "nccl_allreduce": prof["allreduce"][0] / steps,
                                      "voxelgrid_source_tile": prof["voxelgrid"][0] / steps,
                                      "query_sort": prof["query_sort"][0] / steps, "solve": prof["solve"][0] / steps,
                                      "transform_out": prof["transform_out"][0] / steps},
            "setup_ms": setup_ms,
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e / steps, "h2d_bytes_per_step": rec_bytes,
                    "d2h_bytes_per_step": out_bytes + 1024, "aligns_in_flight": depth,
                    **({"pipeline_error": pipeline_error} if pipeline_error else {}),
                    "single_in_flight": {"value": tot_e1 / (ms_e1 * 1e-3), "ms_per_step": ms_e1 / steps},
                    "how": ("host buffers through the C-ABI (set_source H2D, iterate, get_cloud D2H), K steps; "
                            + ("two registration objects on two contexts double-buffer the steps, so one step's PCIe "
                               "copies overlap the other's kernels" if depth == 2 else "one align at a time"))},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}
    if cpu:
        line["cpu_baseline"] = cpu
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 1_000_000


def dump_outputs(d, st, out_dev, with_normals):
    """What the value leg's last align() handed its caller, as .npy files in d: the final transformation, the ICP state
    and the aligned cloud (xyz, and the normals under point-to-plane) -- all rows up to DUMP_ROWS, beyond that the same
    seeded sample of DUMP_ROWS rows on every run, with their row numbers (32 MB at most)."""
    import torch
    os.makedirs(d, exist_ok=True)
    n = int(out_dev.shape[0])
    rows = torch.arange(n) if n <= DUMP_ROWS else torch.from_numpy(
        np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False)))
    cloud = out_dev[rows.to(out_dev.device)].cpu().numpy()
    arrays = {"final_transformation": np.asarray(st["final"], dtype=np.float64),
              "icp_state": np.array([st["converged"], st["state"], st["iterations"], st["n_correspondences"], st["mse"],
                                     st["total_correspondences"]], dtype=np.float64),
              "aligned_xyz": np.ascontiguousarray(cloud[:, 0:3], dtype=np.float32)}
    if with_normals:
        arrays["aligned_normals"] = np.ascontiguousarray(cloud[:, 4:7], dtype=np.float32)
    if n > DUMP_ROWS:
        arrays["aligned_rows"] = rows.numpy().astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


def _protect_stdout():
    """Keep stdout for the ONE JSON line: libraries (NCCL prints its version banner) get stderr instead."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def main():
    global _JSON_OUT
    _JSON_OUT = _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--shard", default="cyclic", choices=["cyclic", "contiguous"],
                    help="strong scaling: Morton chunks dealt round-robin (balanced work) or one contiguous Morton range per rank")
    ap.add_argument("--points", type=int, default=0, help="override the workload's point count (debug / smaller boxes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="e2e leg: one align in flight instead of two")
    ap.add_argument("--no-clocks", action="store_true", help="debug: do not sample clocks during the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (transformation, ICP state, aligned cloud) as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and --steps >= 1 (the reference arm sizes its sample by timing)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
