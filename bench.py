#!/usr/bin/env python
"""bench.py -- points integrated per second on the BASELINE.json workloads (one "step" =
insertPointCloud of one synthetic scan of the named shape).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4] [--impl reference]
                    [--dump-outputs DIR]

Default = BASELINE configs[1] ("config 2": OccupancyMap 2 cm, 131 072-point Velodyne-64-shaped
scan stream, max_range 30 m), the configuration the metric is quoted on; --config 3 (colour map,
2 mm, 640x480 RGB-D, discrete insert) and --config 4 (5 cm, 100 m) time the other single-GPU
configurations the same way.

* value  : whole-job points/s with the scans already resident in HBM (ufo_b200_insert_device,
           async = 1), CUDA events on the map's stream, max over ranks.
* e2e    : the same metric through the reference-facing C-ABI call with HOST (pinned) buffers,
           the way the ROS server drives it (async = 1): every step copies its scan H2D and
           reads back the result counters of a scan D2H inside the timed region; the copy of
           scan k+1 overlaps the kernels of scan k.  e2e.sync is the fully serialised variant
           (wait + read the scan's own counters after every insert).
* sustained: the e2e loop kept running for >= 2 s over the same scans (clock record included).
* roofline: algorithmic bytes (SURVEY.md 8(d) formula on the live device counters) over CUDA-event
           time, against the measured HBM peak: for the dominant kernel and for the whole scan.
           roofline.line_granular: HBM moves whole 128 B lines; the leaf lines the dominant kernel
           touches (counted on the device) and the measured ceiling of that sparse access pattern
           (tools/sector_ceiling.cu -> profiles/r02_sector_ceiling.jsonl).
* cold_start: first scans into a map created with the default pool sizes (pool growth included).
* raycast: voxel visits/s and mark atomics/s of the fused walk against the measured L2 atomic
           ceiling (tools/atomic_ceiling.cu -> profiles/r02_atomic_ceiling.jsonl).
* cpu_baseline / --impl reference: the unmodified reference (oracle/_ref/libufo_ref.so) on a bounded
           sample of the same workload on the host cores.
* --dump-outputs DIR: after the timed steps of `value`, the map they built (voxel keys f64, log-odds
           f32, colour f32; a fixed hash sample above 2^20 voxels) and the last scan's counters, as
           DIR/<name>.npy.  The scans are seeded, so the same arguments feed the same inputs and two
           builds can be compared output for output.

Multi-GPU (torchrun, one rank per GPU): --mode route (default) = ONE scan stream, rays split over
the GPUs, state owned by space, marks forwarded over NVLink peer memory; --mode merge = one sensor
per GPU merged in sensor order (BASELINE config #5); --mode sensors = one sensor stream + map per
GPU (replicas); --mode shard = ONE scan stream broadcast, every GPU walks every ray.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    2: dict(resolution=0.02, max_range=30.0, color=False, discrete=False, kind="velodyne", bricks=1 << 19,
            workload="OccupancyMap 2 cm depth 16, 131072-pt Velodyne-64-shaped synthetic scan stream, max_range 30 m"),
    3: dict(resolution=0.002, max_range=5.0, color=True, discrete=True, kind="rgbd", bricks=1 << 20,
            workload="OccupancyMapColor 2 mm depth 16, 307200-pt RGB-D-shaped synthetic scan stream, max_range 5 m, "
                     "insertPointCloudDiscrete depth 0"),
    4: dict(resolution=0.05, max_range=100.0, color=False, discrete=False, kind="velodyne", bricks=1 << 18,
            workload="OccupancyMap 5 cm depth 16, 131072-pt Velodyne-64-shaped synthetic scan stream, max_range 100 m"),
}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def atomic_ceiling():
    """L2-resident 64-bit reduction throughput measured by tools/atomic_ceiling.cu (G ops/s)."""
    path = os.path.join(ROOT, "profiles", "r02_atomic_ceiling.jsonl")
    best = {}
    try:
        for line in open(path):
            d = json.loads(line)
            if d["pattern"] == "red64_uniform":
                best[d["footprint_mb"]] = d["gops_per_s"]
        return {"l2_resident_gops": best.get(32.0), "at_128mb_gops": best.get(128.0), "source": "profiles/r02_atomic_ceiling.jsonl"}
    except Exception:
        return None


def algorithmic_bytes(st, color=False, p_in=12, part="scan"):
    """SURVEY.md 8(d): N*P_in + U*S_leaf + D1*8*S_leaf + sum_{l>=1} D_l*S_inner + sum_{l>=2} D_l*8*S_inner.
    part="update" keeps the terms the leaf-update kernel (k_update_brick) is responsible for:
    everything except the point input and the levels above the brick (depth >= 5)."""
    s_leaf, s_inner = (8, 12) if color else (4, 8)
    n, u = st["points"], st["touched_voxels"]
    d1, d2, d3, d4, up = (st["touched_octets"], st["touched_blocks"], st["touched_d3"],
                          st["touched_bricks"], st["upper_nodes"])
    if part == "update":
        n, up = 0, 0
    inner_all = d1 + d2 + d3 + d4 + up
    inner_ge2 = d2 + d3 + d4 + up
    return n * p_in + u * s_leaf + d1 * 8 * s_leaf + inner_all * s_inner + inner_ge2 * 8 * s_inner


def sector_ceiling():
    """tools/sector_ceiling.cu: a kernel that does nothing but read-modify-write K3's sector set."""
    path = os.path.join(ROOT, "profiles", "r02_sector_ceiling.jsonl")
    out = {}
    try:
        for line in open(path):
            d = json.loads(line)
            if d["pattern"] in ("k3_leaf", "k3_all"):
                out[d["pattern"] + "_ms"] = d["ms"]
                out[d["pattern"] + "_sectors"] = d["sectors"]
            elif d["pattern"] == "rmw" and d.get("bricks") == "scattered":
                out["rmw_gbs_at_density_%s" % d["density"]] = d["GBps"]
        out["source"] = "profiles/r02_sector_ceiling.jsonl"
        return out
    except Exception:
        return None


def measured_traffic():
    """dram read+write bytes per launch of the dominant kernel from the committed ncu capture."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            return float(d["traffic_bytes_per_launch"]), d["source"]
        except Exception:
            continue
    return None, None


class ClockSampler:
    """SM clock and throttle reasons DURING a timed region.  Sampled in-process through NVML (a thread,
    one query every 5 ms): starting an `nvidia-smi` process next to a 30 ms timed region puts its
    driver initialisation inside that region and can stall kernel launches for tens of ms (seen once
    as a 42 ms hole in the pipelined loop).  Falls back to `nvidia-smi -lms` when pynvml is missing."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    _nvml = None
    _nvml_tried = False
    REASON_BITS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
                   (0x4, "sw_power_cap"))

    @classmethod
    def nvml(cls):
        if not cls._nvml_tried:
            cls._nvml_tried = True
            try:
                import pynvml
                pynvml.nvmlInit()
                cls._nvml = pynvml
            except Exception:
                cls._nvml = None
        return cls._nvml

    def __init__(self, gpu_index, period_ms=5):
        self.path = "/tmp/ufo_clocks_%d_%d.csv" % (os.getpid(), gpu_index)
        self.proc = None
        self.thread = None
        self.gpu = gpu_index
        self.period = period_ms
        self.samples = []

    def _loop(self, nv, handle):
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(handle)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                self.samples.append((float(sm), float(mx), int(rs)))
            except Exception:
                pass
            self._stop.wait(self.period * 1e-3)

    def start(self):
        nv = self.nvml()
        if nv is not None:
            try:
                import threading
                handle = nv.nvmlDeviceGetHandleByIndex(self.gpu)
                self._stop = threading.Event()
                self.thread = threading.Thread(target=self._loop, args=(nv, handle), daemon=True)
                self.thread.start()
                return
            except Exception:
                self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            if self.samples:
                reasons = set()
                for _, _, rs in self.samples:
                    for bit, name in self.REASON_BITS:
                        if rs & bit:
                            reasons.add(name)
                out.update(sm_mhz=float(np.median([x[0] for x in self.samples])),
                           sm_max_mhz=float(max(x[1] for x in self.samples)), samples=len(self.samples),
                           reasons=sorted(reasons), source="nvml")
            return out
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0]))
                    mx.append(float(f[1]))
                except ValueError:
                    continue
                for name, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm), source="nvidia-smi")
        out["reasons"] = sorted(reasons)
        return out


def make_scans(cfg, count, rank):
    """Scans of this rank's sensor: (origins float64, packed clouds, layout, xyz float64 list, rgb list)."""
    from ufomap_b200 import capi, scans
    origins, packed, xyzs, rgbs = [], [], [], []
    layout = capi.XYZ_F32
    base = scans.sensor_ring(rank, 8) if rank else None
    for k in range(count):
        rgb = None
        if cfg["kind"] == "rgbd":
            if rank == 0:
                o, p, rgb = scans.rgbd(k=k)
            else:
                o, p, rgb = scans.rgbd(k=k, origin=np.array([0.0013 + 0.02 * k, 0.0021 + 0.01 * k + 0.5 * rank, 0.0007]))
        elif rank == 0:
            o, p = scans.velodyne64(k=k)
        else:
            o = base + np.array([0.25 * k, 0.10 * k, 0.0])
            o, p = scans.velodyne64(k=k, origin=o, seed=88172645463325252 + 7919 * rank)
        buf, layout = capi.pack_points(p, rgb, np.float32)
        origins.append(o)
        packed.append(np.ascontiguousarray(buf))
        xyzs.append(p)
        rgbs.append(rgb)
    return origins, packed, layout, xyzs, rgbs


def route_slice(n_pts, rank, world, columns=2048):
    """Rays of `rank` in the routed mode: a contiguous azimuth sector of every ring (ring-major
    scan of `columns` azimuths per ring): neighbouring rays share bricks, so a rank's marks stay
    mostly in bricks only it touches and little has to cross GPUs."""
    if n_pts % columns:
        return np.arange(rank, n_pts, world)
    az = np.arange(n_pts) % columns
    lo, hi = rank * columns // world, (rank + 1) * columns // world
    return np.nonzero((az >= lo) & (az < hi))[0]


def max_over_ranks(value, world, device=None):
    """MAX-reduce a per-rank scalar (the timed region of the slowest rank is the job's time)."""
    if world <= 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _ref_class():
    import oracle_lib
    kind = "reference" if oracle_lib.have_ref() else "port"
    if kind == "port":
        oracle_lib.build_oracle()
    return kind, (oracle_lib.RefMap if kind == "reference" else oracle_lib.OracleMap)


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's own CPU insertPointCloud on the host cores, each step a
    bounded sample (every `stride`-th point of scan k) of the same workload.  The stride starts at
    4 (config 3: 64, the reference cannot hold denser 2 mm scans in memory) and is doubled if the
    projected run would exceed --ref-budget seconds."""
    if rank != 0:
        return
    kind, cls = _ref_class()
    stride = 64 if args.config == 3 else 4
    total = args.steps + args.warmup
    origins, _, _, xyzs, rgbs = make_scans(cfg, total, 0)
    m = cls(cfg["resolution"], color=cfg["color"])
    times, strides, npts = [], [], []
    t_start = time.time()
    for k in range(total):
        elapsed = time.time() - t_start
        if k >= 1 and elapsed / k * total > args.ref_budget and stride < 64:
            stride *= 2
        pts = xyzs[k][::stride]
        rgb = rgbs[k][::stride] if rgbs[k] is not None else None
        secs = m.insert(origins[k], pts, rgb=rgb, max_range=cfg["max_range"], discrete=cfg["discrete"])
        if k >= args.warmup:
            times.append(secs)
            strides.append(stride)
            npts.append(len(pts))
    t = float(np.sum(times))
    value = float(np.sum(npts)) / t
    sample = "every %s-th point of each scan (%d..%d pts/step)" % (
        "/".join(str(s) for s in sorted(set(strides))), min(npts), max(npts))
    line = {
        "impl": "reference", "metric": "points_integrated_per_s", "value": value, "unit": "points/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 geometry + f32 log-odds", "data": "synthetic",
        "config": {"workload": cfg["workload"], "sample": sample},
        "same_config": False, "sample_stride": sorted(set(strides)),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": 2, "kind": kind,
                         "sample": "insertPointCloud of %s of scans %d..%d, one map, async=false; the reference uses "
                                   "1 caller + 1 hit thread of %d host cores" % (sample, args.warmup, total - 1, os.cpu_count() or 0)},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(cfg, origins, xyzs, rgbs):
    """Bounded CPU sample for the main line: ~10-30 s of the reference on scan 0 and 1."""
    kind, cls = _ref_class()
    stride = 64 if cfg["kind"] == "rgbd" else 16
    m = cls(cfg["resolution"], color=cfg["color"])
    secs, npts = 0.0, 0
    for k in range(2):
        pts = xyzs[k][::stride]
        rgb = rgbs[k][::stride] if rgbs[k] is not None else None
        t = m.insert(origins[k], pts, rgb=rgb, max_range=cfg["max_range"], discrete=cfg["discrete"])
        if k >= 1:  # scan 0 warms allocator and hash tables (BASELINE.md section 4)
            secs += t
            npts += len(pts)
    m.close()
    return {"value": npts / secs, "unit": "points/s", "cores": 2, "kind": kind,
            "sample": "insertPointCloud of every %d-th point (%d pts) of scan 1 after scan 0 as warm-up, "
                      "async=false, 1 caller + 1 hit thread of %d host cores" % (stride, npts, os.cpu_count() or 0)}


DUMP_MAX_VOXELS = 1 << 20   # 40 B a voxel at most (keys f64, log-odds f32, colour f32): 40 MB
COUNTER_NAMES = ("points", "rays", "touched_voxels", "hit_voxels", "touched_octets", "touched_lines",
                 "touched_blocks", "touched_d3", "touched_bricks", "upper_nodes", "blocks_in_map", "bricks_in_map")


def dump_outputs(out_dir, m, color, prefix=""):
    """What the timed insert path leaves a caller: the map's value field (every voxel with a
    non-default payload) and the result counters of the last scan, as .npy files in `out_dir`.
    A field of more than DUMP_MAX_VOXELS voxels is sampled by a fixed hash of the voxel code, so
    two builds that computed the same field write the same sample."""
    os.makedirs(out_dir, exist_ok=True)
    m.wait()
    codes, occ, rgb = m.value_field(sort=False)
    if len(codes) > DUMP_MAX_VOXELS:
        mixed = codes * np.uint64(0x9E3779B97F4A7C15)   # wraps: a fixed bijective hash of the code
        keep = mixed < np.uint64(int(2.0 ** 64 * DUMP_MAX_VOXELS / len(codes)))
        codes, occ, rgb = codes[keep], occ[keep], rgb[keep]
    order = np.argsort(codes, kind="stable")
    codes, occ, rgb = codes[order], occ[order], rgb[order]
    keys = np.zeros((len(codes), 3), np.float64)   # the depth-0 key: code bits interleaved x, y, z
    for i in range(21):
        for a in range(3):
            keys[:, a] += ((codes >> np.uint64(3 * i + a)) & np.uint64(1)).astype(np.float64) * float(1 << i)
    st = m.stats()
    arrays = {"voxel_keys": keys, "log_odds": occ.astype(np.float32),
              "scan_counters": np.array([float(st[k]) for k in COUNTER_NAMES], np.float64)}
    if color:
        arrays["rgb"] = rgb.astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of the sustained e2e loop (0: skip)")
    ap.add_argument("--ref-budget", type=float, default=1200.0, help="--impl reference: wall-clock budget in seconds")
    ap.add_argument("--mode", default="route", choices=["route", "merge", "sensors", "shard"],
                    help="N>1: 'route' (default) = ONE scan stream, rays split over the GPUs, space-owned state, "
                         "foreign marks written to the owners over NVLink peer memory (strong scaling, SURVEY.md "
                         "8(e) variant 2); 'merge' = one sensor per GPU, owners apply the sensors in sensor order "
                         "(BASELINE config #5, weak scaling); 'sensors' = independent replicas (one sensor stream + "
                         "map per GPU, no merge); 'shard' = one stream broadcast, every GPU walks every ray and "
                         "keeps its own bricks (variant 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of `value`, write the map's value field (sampled above %d voxels) "
                         "and the last scan's counters to DIR/<name>.npy" % DUMP_MAX_VOXELS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    cfg = CONFIGS[args.config]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    from ufomap_b200 import capi

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    total = args.steps + args.warmup
    mode = args.mode if world > 1 else "single"
    if mode in ("route", "merge") and (cfg["color"] or cfg["discrete"]):
        mode = "sensors"  # routed passes: mono maps, plain insertion
    shard = mode == "shard"
    routed = mode in ("route", "merge")
    one_stream = mode in ("route", "shard")
    origins, packed, layout, xyzs, rgbs = make_scans(cfg, total, 0 if one_stream else rank)
    n_pts = packed[0].shape[0]
    p_in = packed[0].nbytes // n_pts
    if mode == "route":
        # this rank's rays: an azimuth sector of every ring (the scan is ring-major, 2048 columns)
        idx = route_slice(n_pts, rank, world)
        packed = [np.ascontiguousarray(c[idx]) for c in packed]
    n_mine = packed[0].shape[0]
    stream = torch.cuda.current_stream(dev)
    ins_kw = dict(max_range=cfg["max_range"], discrete=cfg["discrete"])
    token = torch.zeros(1, device=dev) if routed else None
    opened = []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def fresh_map():
        m = capi.Map(cfg["resolution"], color=cfg["color"], device=local_rank, initial_bricks=cfg["bricks"])
        m.set_stream(stream.cuda_stream)
        if shard:
            m.set_shard(rank, world)
        if routed:
            # inboxes: one cudaIpc handle per rank through the control plane, mapped by every peer
            ptr = m.route_setup(rank, world, cap_bricks=max(1 << 16, 400000 // world), cap_hits=1 << 18)
            handles = [None] * world
            dist.all_gather_object(handles, capi.ipc_export(ptr))
            peers = [ptr if r == rank else capi.ipc_open(handles[r]) for r in range(world)]
            opened.extend(p for r, p in enumerate(peers) if r != rank)
            m.route_connect(peers)
            dist.barrier()
        return m

    def close_map(m):
        m.wait()
        if routed:
            dist.barrier()  # nobody writes into a peer inbox any more
            while opened:
                capi.ipc_close(opened.pop())
            dist.barrier()
        m.close()

    def routed_step(mm, k, ptr, on_device):
        mm.route_mark(origins[k], ptr, n_mine, layout, max_range=cfg["max_range"], on_device=on_device,
                      self_too=(mode == "merge"))
        dist.all_reduce(token)  # the barrier between forwarding and applying, ordered on the map's stream
        if mode == "merge":
            for s_ in range(world):
                mm.route_apply(s_, 1, s_ == world - 1)
        else:
            mm.route_apply(0, world, True)

    def timed_loop(m, feed, first, count, sync_each=False):
        """`count` steps starting at scan index `first`; returns (ms, per-scan stats, launches, clocks)."""
        m.wait()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        per_scan, launches = [], 0
        e0.record(stream)
        for k in range(first, first + count):
            feed(m, k % total)
            # D2H of a scan's counters (the step's result): of this scan (sync_each) or, pipelined,
            # of the previous one while this one runs
            st = m.stats() if sync_each else m.completed_stats()
            if st["points"]:
                per_scan.append(st)
                launches += st["launches"]
        m.wait()
        e1.record(stream)
        barrier()
        clocks = sampler.stop()
        ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
        if not sync_each:
            per_scan.append(m.stats())
            per_scan = per_scan[-count:]
        launches = sum(s["launches"] for s in per_scan)
        return ms, per_scan, launches, clocks

    # ---- device-resident inputs: `value` ---------------------------------
    d_clouds = [torch.from_numpy(c).to(dev) for c in packed]
    torch.cuda.synchronize(dev)
    m = fresh_map()
    m.set_profiling(1)
    bcast = torch.empty_like(d_clouds[0]) if shard else None

    def feed_device(mm, k):
        src = d_clouds[k]
        if routed:
            routed_step(mm, k, src.data_ptr(), True)
            return
        if shard:
            # the one collective of the sharded mode: rank 0's scan goes to every GPU
            if rank == 0:
                bcast.copy_(src)
            dist.broadcast(bcast, src=0)
            src = bcast
        mm.insert_packed(origins[k], src.data_ptr(), n_mine, layout, on_device=True, async_=True, **ins_kw)

    for k in range(args.warmup):
        feed_device(m, k)
    ms_dev, per_scan, launches, clocks = timed_loop(m, feed_device, args.warmup, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m, cfg["color"], "rank%d_" % rank if world > 1 else "")
    dev_bytes = per_scan[-1]["device_bytes"]
    # one more scan with visit / mark counting switched on (not timed): raycast counters
    m.set_profiling(2)
    feed_device(m, total - 1)
    counted = m.stats()
    close_map(m)
    del d_clouds
    torch.cuda.empty_cache()

    # ---- host buffers through the C ABI: `e2e` -----------------------------
    h_clouds = [torch.from_numpy(c).pin_memory() for c in packed]
    m = fresh_map()
    stage = torch.empty_like(torch.from_numpy(packed[0]), device=dev) if shard else None

    def feed_host(mm, k):
        if routed:
            routed_step(mm, k, h_clouds[k].data_ptr(), False)
            return
        if shard:
            if rank == 0:
                stage.copy_(h_clouds[k], non_blocking=True)  # H2D once, on rank 0
            dist.broadcast(stage, src=0)
            mm.insert_packed(origins[k], stage.data_ptr(), n_pts, layout, on_device=True, async_=True, **ins_kw)
            return
        mm.insert_packed(origins[k], h_clouds[k].data_ptr(), n_mine, layout, on_device=False, async_=True, **ins_kw)

    for k in range(args.warmup):
        feed_host(m, k)
    ms_e2e, e2e_scans, _, clocks_e2e = timed_loop(m, feed_host, args.warmup, args.steps)
    d2h = int(e2e_scans[-1]["result_bytes"])
    # fully serialised variant on a fresh map (same scans)
    close_map(m)
    m = fresh_map()
    for k in range(args.warmup):
        feed_host(m, k)
    ms_sync, _, _, _ = timed_loop(m, feed_host, args.warmup, args.steps, sync_each=True)
    # sustained: keep the pipelined e2e loop running for >= args.sustain seconds over the same scans
    sustained = None
    if args.sustain > 0:
        est = max(ms_e2e / args.steps, 1e-3)
        count = int(args.sustain * 1e3 / est) + 1
        ms_sus, _, _, clocks_sus = timed_loop(m, feed_host, 0, count)
        streams_ = 1 if one_stream else world
        sustained = {"seconds": ms_sus * 1e-3, "steps": count, "value": streams_ * count * n_pts / (ms_sus * 1e-3),
                     "unit": "points/s", "ms_per_step": ms_sus / count, "clocks": clocks_sus,
                     "note": "scans cycle through the same %d poses (the map stops growing; work per scan unchanged)" % total}
    close_map(m)

    # cold start: a map created with the DEFAULT pool sizes integrates its first scans, device pools
    # growing on the way (allocation, copy, scan repeated): what the pre-sized pools of the timed loops
    # leave out.  Wall clock, single GPU modes only.
    cold = None
    if rank == 0 and not routed and not shard:
        try:
            mc = capi.Map(cfg["resolution"], color=cfg["color"], device=local_rank)
            t0 = time.perf_counter()
            mc.insert_packed(origins[0], h_clouds[0].data_ptr(), n_mine, layout, on_device=False, async_=False, **ins_kw)
            t1 = time.perf_counter()
            st0 = mc.stats()
            mc.insert_packed(origins[1], h_clouds[1].data_ptr(), n_mine, layout, on_device=False, async_=False, **ins_kw)
            t2 = time.perf_counter()
            st1 = mc.stats()
            cold = {"first_scan_ms": (t1 - t0) * 1e3, "first_scan_regrows": int(st0["regrows"]),
                    "second_scan_ms": (t2 - t1) * 1e3, "second_scan_regrows": int(st1["regrows"]),
                    "note": "default pool sizes, wall clock incl. pool growth and repeated marking; not part of value / e2e"}
            mc.close()
        except Exception as exc:  # never let the side measurement take the bench line down
            cold = {"error": str(exc)[:200]}

    steps = args.steps
    streams = 1 if one_stream else world  # route / shard integrate ONE stream with all GPUs
    value = streams * steps * n_pts / (ms_dev * 1e-3)
    e2e = streams * steps * n_pts / (ms_e2e * 1e-3)
    e2e_sync = streams * steps * n_pts / (ms_sync * 1e-3)

    # roofline of the device work of one insert (K1..K4), averaged over the timed scans
    peak, peak_src = measured_peak()
    color = cfg["color"]
    alg = float(np.mean([algorithmic_bytes(s, color, p_in) for s in per_scan]))
    alg_upd = float(np.mean([algorithmic_bytes(s, color, p_in, part="update") for s in per_scan]))
    t_scan_ms = float(np.mean([s["ms_total"] for s in per_scan]))
    kern = {k: float(np.mean([s[k] for s in per_scan])) for k in
            ("ms_h2d", "ms_points", "ms_rays", "ms_scatter", "ms_update", "ms_propagate")}
    achieved = alg_upd / (kern["ms_update"] * 1e-3) / 1e9
    pipeline = alg / (t_scan_ms * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic()
    lines = float(np.mean([s.get("touched_lines", 0) for s in per_scan]))
    last = per_scan[-1]
    ceil = atomic_ceiling()
    t_walk = (kern["ms_rays"] + kern["ms_scatter"]) * 1e-3
    raycast = {"kernel": "k_split + k_walk_mark (fused exact FP64 walk + mask reductions)", "ms": t_walk * 1e3,
               "visits": int(counted["visits"]), "visits_per_s": counted["visits"] / t_walk if t_walk else None,
               "l2_atomic_ceiling": ceil}

    if rank == 0:
        line = {
            "metric": "points_integrated_per_s", "value": value, "unit": "points/s",
            "scans_per_s": value / n_pts, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "strong" if one_stream else "weak",
            "vs_baseline": None, "dtype": "f64 geometry + f32 log-odds", "data": "synthetic",
            "config": {"workload": cfg["workload"], "points_per_scan": n_pts,
                       "input": "float32 xyz" + (" + rgb" if color else ""),
                       "parallelism": {
                           "single": "1 map on 1 GPU",
                           "route": "ONE scan stream; rays split over the GPUs by azimuth sector, state owned by space "
                                    "(hash of the 16^3 brick), foreign brick masks / hit voxels written into the "
                                    "owner's inbox over NVLink peer memory, one 4-byte NCCL all-reduce as barrier",
                           "merge": "one sensor per GPU (BASELINE config #5 shape); owners apply the sensors' marks in "
                                    "sensor order; marks forwarded over NVLink peer memory",
                           "shard": "one scan stream broadcast over NCCL, every GPU walks every ray, map sharded by brick ownership",
                           "sensors": "one sensor stream + map per GPU, no merge (independent replicas)"}[mode],
                       "mode": mode,
                       "l2": "per-scan working set (%.1f GB leaf data touched, map %.1f GB) exceeds the 126 MB L2; no flush"
                             % (last["touched_blocks"] * (512 if color else 256) / 1e9, dev_bytes / 1e9)},
            "e2e": {"value": e2e, "unit": "points/s", "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": int(n_mine * p_in), "d2h_bytes_per_step": d2h,
                    "mode": "async=1 (server default): H2D of scan k+1 overlaps the kernels of scan k",
                    "regrows": int(sum(s_["regrows"] for s_ in e2e_scans)),
                    "max_scan_device_ms": float(max(s_["ms_total"] for s_ in e2e_scans)),
                    "sync": {"value": e2e_sync, "ms_per_step": ms_sync / steps,
                             "mode": "wait + read the scan's own counters after every insert"}},
            "sustained": sustained,
            "cold_start": cold,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": "k_update_brick: hit/miss log-odds update of the marked voxels and depth 1-4 "
                                   "aggregates over the scan's touched bricks; CUDA events on the map's stream "
                                   "around every launch of the timed region",
                         "algorithmic_bytes_per_launch": alg_upd, "ms_per_launch": kern["ms_update"],
                         "traffic_source": traffic_src,
                         # HBM moves whole 128 B lines (profiles/r02_sector_ceiling.jsonl: sparse 32 B sectors
                         # cost what their lines cost): the leaf lines K3 touches, read + written, over its time
                         "line_granular": {"leaf_lines_128B": lines, "leaf_line_bytes": lines * 256.0,
                                           "leaf_line_gbs": lines * 256.0 / (kern["ms_update"] * 1e-3) / 1e9,
                                           "frac_of_peak_leaf_lines_only": lines * 256.0 / (kern["ms_update"] * 1e-3) / 1e9 / peak,
                                           "sector_ceiling": sector_ceiling()},
                         # SURVEY.md 8(d)'s whole-pipeline figure: all algorithmic bytes of a scan over the
                         # device time of the whole insert (K1..K4)
                         "pipeline": {"algorithmic_bytes_per_scan": alg, "device_ms_per_scan": t_scan_ms,
                                      "achieved": pipeline, "frac": pipeline / peak}},
            "raycast": raycast,
            "kernels_ms": kern,
            "counters": {k: int(last[k]) for k in ("rays", "touched_voxels", "hit_voxels", "touched_octets", "touched_lines",
                                                    "touched_blocks", "touched_d3", "touched_bricks",
                                                    "upper_nodes", "blocks_in_map", "bricks_in_map", "regrows")},
            "gpu_launches": int(launches),
            "clocks": clocks, "clocks_e2e": clocks_e2e,
        }
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_baseline_sample(cfg, origins, xyzs, rgbs)
            except Exception as e:  # the checker is optional for the GPU number
                line["cpu_baseline"] = {"value": None, "error": str(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
