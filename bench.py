#!/usr/bin/env python
"""Benchmark of the hot path: integrated points/s of MergedTsdfIntegrator on 640x480
scans at 0.05 m voxels (BASELINE.json's metric), one scan per step.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our engine (one JSON line)
  python bench.py ... --dump-outputs DIR                       ... and the resulting map as DIR/*.npy
  python bench.py --impl reference ...                         the reference's own CPU
                                                               MergedTsdfIntegrator (oracle/_ref)
Multi-GPU runs are launched by torchrun, one rank per GPU (DESIGN.md "multi-GPU").

JSON keys follow the driver's contract; see DESIGN.md "measurement" for how value, e2e,
roofline and cpu_baseline are produced.
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

# The pipelined path keeps ~18 CUDA streams busy (front lanes, their side streams, walk, sorts, apply, copies).
# By default a process gets 8 hardware work queues and streams beyond that share them, which serialises
# kernels that could overlap; the variable must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "integrated points/sec (640x480 scan, 0.05 m voxel)"

# The workloads of BASELINE.json / SURVEY.md section 8(d).  "bench" is the configuration the metric is
# quoted on (Merged, 640x480, 0.05 m voxels, truncation 4 voxels: the C3 / C4 cloud stream through the
# Merged integrator) and the only one the driver runs; the others are selected with --config and are
# what BASELINE.md's table is filled from.
CONFIGS = {
    "bench": dict(workload="merged_640x480_room_sequence_0.05m", kind="merged", voxel=0.05, scan="c3_room_scan",
                  cfg=dict(default_truncation_distance=0.2), opts=dict(max_blocks=16384, max_points_per_scan=1 << 19,
                                                                       max_updates_per_pass=1 << 24),
                  scan_text="640x480 pinhole, box room + 4 objects, 15% dropouts, 30 Hz handheld trajectory"),
    "C1": dict(workload="C1_simple_64x48_planar_wall_0.20m", kind="simple", voxel=0.2, scan="c1_planar_wall",
               cfg=dict(default_truncation_distance=0.8), opts=dict(max_blocks=4096, max_points_per_scan=1 << 16,
                                                                    max_updates_per_pass=1 << 22),
               scan_text="64x48 pinhole, planar wall at 3 m (the same scan every step)"),
    "C2": dict(workload="C2_merged_640x480_sphere_room_0.10m", kind="merged", voxel=0.1, scan="c2_sphere_scan",
               cfg=dict(default_truncation_distance=0.4), opts=dict(max_blocks=16384, max_points_per_scan=1 << 19,
                                                                    max_updates_per_pass=1 << 24),
               scan_text="640x480 pinhole inside a 3 m sphere, 300-scan orbit (truncation 4 voxels; --trunc 4.0 for the literal 4 m)"),
    "C3": dict(workload="C3_fast_640x480_room_sequence_0.05m", kind="fast", voxel=0.05, scan="c3_room_scan",
               cfg=dict(default_truncation_distance=0.2), opts=dict(max_blocks=16384, max_points_per_scan=1 << 19,
                                                                    max_updates_per_pass=1 << 26),
               scan_text="640x480 pinhole, box room + 4 objects, 15% dropouts, 30 Hz handheld trajectory"),
    "C4": dict(workload="C4_merged_plus_esdf_640x480_0.05m", kind="merged", voxel=0.05, scan="c3_room_scan", esdf=True,
               cfg=dict(default_truncation_distance=0.2), opts=dict(max_blocks=16384, max_points_per_scan=1 << 19,
                                                                    max_updates_per_pass=1 << 24),
               scan_text="as bench, EsdfIntegrator::updateFromTsdfLayer(true) after every scan (ROS defaults)"),
    "C5": dict(workload="C5_merged_lidar_2048x128_0.05m", kind="merged", voxel=0.05, scan="c5_lidar_scan",
               cfg=dict(default_truncation_distance=0.2, max_ray_length_m=10.0, use_const_weight=1),
               opts=dict(max_blocks=16384, max_points_per_scan=1 << 19, max_updates_per_pass=1 << 25),
               scan_text="2048x128 spinning LiDAR in a 9x9x4 m hall with pillars, ~13 M voxel updates per scan"),
}
KIND_ID = {"simple": 1, "merged": 2, "fast": 3}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def make_scans(conf, n, start=0):
    from voxblox_b200 import scenes

    if conf["scan"] == "c1_planar_wall":
        s = scenes.c1_planar_wall()
        return [s for _ in range(n)]
    return scenes.generate_parallel(getattr(scenes, conf["scan"]), range(start, start + n))


def config_dict(conf, scans_timed):
    """The `config` object of the JSON line: identical in our arm and in the reference arm."""
    n_mean = float(np.mean([int(s[0].shape[0]) for s in scans_timed])) if scans_timed else 0.0
    return {"workload": conf["workload"], "integrator": conf["kind"], "voxel_size_m": conf["voxel"],
            "truncation_m": conf["cfg"]["default_truncation_distance"], "voxels_per_side": 16,
            "scan": conf["scan_text"], "points_per_scan_mean": n_mean,
            "l2": "every step integrates a different scan (cloud set > L2); the map's voxel blocks stay hot across "
                  "steps as they do in a mapping session"}


# ------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  The timed region of this workload is
    tens of milliseconds, shorter than one `nvidia-smi -lms` period, so the sampler reads the same
    counters through NVML (nvidia-ml-py) from a thread every ~2 ms; rows are time-stamped and only
    those inside [mark_begin, mark_end] are reported (falling back to nvidia-smi rows if NVML is
    unavailable)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index=0):
        self.rows = []      # (t, sm_mhz, max_mhz, reasons bitmask)
        self.proc = None
        self.index = index
        self.stop_flag = False
        self.thread = None
        self.source = None
        self.t_begin = self.t_end = None

    def _nvml_loop(self, nv, h):
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                rs = int(get_reasons(h)) if get_reasons else 0
                self.rows.append((time.perf_counter(), float(sm), float(mx) if mx else None, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.index
            if vis:
                try:
                    phys = int(vis.split(",")[self.index])
                except Exception:
                    phys = self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.source = "nvml"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.source = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                rs = 0
                for nme, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                    if v.lower().startswith("active"):
                        rs |= self.BITS[nme]
                self.rows.append((time.perf_counter(), float(f[0]), float(f[1]), rs))
            except ValueError:
                continue

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi / NVML unavailable"]}
        if self.t_end is None:
            self.t_end = time.perf_counter()
        self.stop_flag = True
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.thread:
            self.thread.join(timeout=1)
        t0 = self.t_begin if self.t_begin is not None else -1e30
        inside = [r for r in self.rows if t0 <= r[0] <= self.t_end]
        window = "timed region"
        if not inside and self.rows:
            # nothing landed inside a very short region: take the sample nearest to it
            mid = 0.5 * (t0 + self.t_end)
            inside = [min(self.rows, key=lambda r: abs(r[0] - mid))]
            window = "nearest sample to the timed region"
        sm = [r[1] for r in inside]
        mx = [r[2] for r in inside if r[2]]
        bits = 0
        for r in inside:
            bits |= r[3]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(k for k, b in self.BITS.items() if bits & b),
                "source": self.source, "window": window}


# -------------------------------------------------------------------- CPU baseline
def time_reference(conf, scans, threads, which=None, esdf=False):
    """Seconds inside integratePointCloud per scan (stopwatch placed like
    voxblox_ros/src/tsdf_server.cc:305-307) for the CPU implementation."""
    from oracle import pyoracle as po

    which = which or ("reference" if po.available("reference") else "port")
    lib = po.OracleLib(which)
    cfg = po.TsdfConfig(integrator_threads=threads, **conf["cfg"])
    m = po.OracleMap(lib, cfg, conf["voxel"], 16)
    if esdf:
        m.esdf_create(po.EsdfConfig(max_distance_m=2.0, default_distance_m=2.0,
                                    min_distance_m=conf["cfg"]["default_truncation_distance"] / 2, min_diff_m=1e-3))
    secs = []
    for s in scans:
        m.integrate(KIND_ID[conf["kind"]], s)
        t = m.last_seconds()
        if esdf:
            m.esdf_update(batch=False, clear_updated_flag=True)
            t += m.last_seconds()
        secs.append(t)
    m.close()
    return which, secs


def calibrate_threads(conf, scans):
    """The reference defaults to hardware_concurrency threads (tsdf_integrator.h:70) but
    its per-call std::thread fan-out often loses to fewer threads; give it the best."""
    ncpu = os.cpu_count() or 1
    cands = sorted({1, 4, 8, 16, min(32, ncpu), ncpu})
    best = None
    detail = {}
    for t in cands:
        if t > ncpu:
            continue
        _, secs = time_reference(conf, scans, t)
        v = float(np.mean(secs[1:])) if len(secs) > 1 else secs[0]
        detail[str(t)] = round(v * 1e3, 3)
        if best is None or v < best[1]:
            best = (t, v)
    return best[0], detail


def run_reference_arm(args, conf, rank):
    """The reference's own CPU implementation of the path (oracle/_ref: its translation units compiled
    where they lie) on this box's host cores; none of the engine is loaded in this process."""
    if rank != 0:
        return
    scans = make_scans(conf, args.warmup + args.steps)
    threads, detail = calibrate_threads(conf, scans[:3])
    which, secs = time_reference(conf, scans, threads, esdf=bool(conf.get("esdf")))
    timed = secs[args.warmup:]
    pts = sum(int(s[0].shape[0]) for s in scans[args.warmup:])
    total = float(sum(timed))
    value = pts / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, len(timed)),
        "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(conf, scans[args.warmup:]),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": which,
                         "sample": f"{len(timed)} scans of the workload; {conf['kind']} integrator, integrator_threads={threads} "
                                   f"(fastest of {detail} ms/scan; host has {os.cpu_count()} logical cores)"},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------- DRAM traffic (ncu)
NCU_METRICS = "dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum"


def traffic_child(conf):
    """Run under `ncu` by measure_traffic(): a few synchronous scans, nothing else."""
    import torch

    import voxblox_b200 as vb

    scans = make_scans(conf, 5)
    layer = vb.Layer(conf["voxel"], 16, engine_options=vb.EngineOptions(**conf["opts"]))
    integ = vb.TsdfIntegratorFactory.create(conf["kind"], vb.TsdfIntegratorConfig(**conf["cfg"]), layer)
    d = [(torch.from_numpy(s[0]).cuda(), torch.from_numpy(s[1]).cuda()) for s in scans]
    for s, (x, c) in zip(scans, d):
        integ.integratePointCloudDevice((s[2], s[3]), x.data_ptr(), c.data_ptr(), int(s[0].shape[0]))
    print(json.dumps({"scans": len(scans)}), flush=True)


def measure_traffic(conf_name, timeout_s=300, cache_control="all"):
    """dram__bytes_read.sum + dram__bytes_write.sum per kernel, measured NOW on this box by running a
    5-scan child of this script under ncu.  cache_control "all" (ncu's default) flushes the caches before
    every kernel: an upper bound in which every intermediate buffer (sort ping-pong, records, ray tables)
    is charged as DRAM traffic although the pipeline hands it from kernel to kernel through the 126 MB L2;
    "none" leaves the caches alone, so a kernel finds what the previous kernel wrote where the real run
    finds it.  Returns bytes per scan per kernel name, or {"unavailable": why}."""
    import csv
    import shutil
    import tempfile

    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return {"unavailable": "ncu not found"}
    with tempfile.TemporaryDirectory() as td:
        logf = os.path.join(td, "ncu.csv")
        cmd = [ncu, "--metrics", NCU_METRICS, "--clock-control", "none", "--cache-control", cache_control,
               "--print-units", "base", "--csv", "--log-file", logf, sys.executable, os.path.abspath(__file__), "--traffic-child", "--config", conf_name]
        try:
            env = dict(os.environ)
            env.pop("RANK", None)
            env.pop("WORLD_SIZE", None)
            p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout_s, env=env)
        except Exception as exc:
            return {"unavailable": f"ncu run failed: {exc!r}"}
        if p.returncode != 0 or not os.path.exists(logf):
            return {"unavailable": f"ncu exit code {p.returncode}: {p.stderr[-300:]}"}
        n_scans = 5
        per = {}
        with open(logf, newline="") as f:
            rows = [r for r in csv.reader(f) if len(r) > 10]
        if not rows:
            return {"unavailable": "ncu wrote no rows"}
        hdr = None
        for r in rows:
            if "Kernel Name" in r and "Metric Name" in r:
                hdr = r
                continue
            if hdr is None:
                continue
            rec = dict(zip(hdr, r))
            name = rec.get("Kernel Name", "").split("(")[0].split("<")[0].replace("void ", "").split("::")[-1]
            try:
                val = float(rec.get("Metric Value", "0").replace(",", ""))
            except ValueError:
                continue
            d = per.setdefault(name, {"dram_bytes": 0.0, "ns": 0.0, "launches": 0})
            m = rec.get("Metric Name", "")
            if m.startswith("dram__bytes"):
                d["dram_bytes"] += val
            elif m.startswith("gpu__time_duration"):
                d["ns"] += val
                d["launches"] += 1
        out = {k: {"dram_bytes_per_scan": v["dram_bytes"] / n_scans, "us_per_scan_under_ncu": v["ns"] / n_scans / 1e3,
                   "launches_per_scan": v["launches"] / n_scans} for k, v in per.items()}
        return {"per_kernel": out, "total_dram_bytes_per_scan": sum(v["dram_bytes"] for v in per.values()) / n_scans,
                "scans": n_scans, "how": "ncu --metrics " + NCU_METRICS + " --cache-control " + cache_control +
                ("  (caches flushed before every kernel)" if cache_control == "all" else
                 "  (caches left as the previous kernel left them, as in the real run)") + ", run inside this bench"}


# ------------------------------------------------------------------ output dump
DUMP_MAX_BLOCKS = 384   # sampled blocks: 4096 voxels x (4 + 4 + 16 B TSDF + 8 B ESDF) each, ~48 MB in all


def dump_outputs(out_dir, layer, esdf_layer=None):
    """The map a caller of the timed path holds after its last step, as .npy files: every allocated block index
    and, for a seeded sample of at most DUMP_MAX_BLOCKS of those blocks (all of them when there are fewer), the
    voxels.  Block indices are sorted, so two builds with the same map dump the same sample."""
    os.makedirs(out_dir, exist_ok=True)

    def save(name, a, dtype):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=dtype))

    for prefix, lay in (("tsdf", layer), ("esdf", esdf_layer)):
        if lay is None:
            continue
        idx = lay.getAllAllocatedBlocks()
        pick = np.arange(len(idx))
        if len(idx) > DUMP_MAX_BLOCKS:
            pick = np.sort(np.random.default_rng(0).choice(len(idx), DUMP_MAX_BLOCKS, replace=False))
        vox, upd = lay.getBlocks(idx[pick])
        save(prefix + "_block_indices", idx, np.float64)
        save(prefix + "_sample_block_indices", idx[pick], np.float64)
        save(prefix + "_sample_updated", upd, np.float32)
        save(prefix + "_sample_distance", vox["distance"], np.float32)
        if prefix == "tsdf":
            save("tsdf_sample_weight", vox["weight"], np.float32)
            save("tsdf_sample_color", vox["color"], np.float32)
        else:
            save("esdf_sample_observed", vox["observed"], np.float32)


# --------------------------------------------------------------------------- ours
STAGE_OF_KERNEL = {  # stage name (Layer.stageMs) -> kernels that run in it
    "point_keys": ("k_point_bounds", "k_point_keys"), "point_sort": ("k_sort",),
    "update_sort": ("k_sort",), "bundle_order": ("k_order_prefix", "k_order_heads", "k_bundle_order"),
    "bundle_merge": ("k_merge",), "scan": ("k_exclusive_scan",),
    "ray_emit": ("k_rays_emit_warp", "k_rays_emit", "k_rays_count"), "assign": ("k_assign",),
    "apply": ("k_apply_short", "k_apply_verify", "k_apply_long"),
}


def run_ours(args, conf, rank, world):
    import torch
    import torch.distributed as dist

    import voxblox_b200 as vb
    from voxblox_b200 import sharded

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_total = args.warmup + args.steps
    # N > 1: ONE map, sharded over the ranks by block ownership; every rank receives every scan
    # (identical, seeded) -- strong scaling.  DESIGN.md "multi-GPU".
    scans = make_scans(conf, n_total)
    npts = [int(s[0].shape[0]) for s in scans]
    cfg = vb.TsdfIntegratorConfig(**conf["cfg"])
    kind = conf["kind"]
    do_esdf = bool(conf.get("esdf"))

    def fresh(rank_=rank, world_=world):
        opts = vb.EngineOptions(device=local, rank=rank_, world_size=world_, **conf["opts"])
        layer = vb.Layer(conf["voxel"], 16, engine_options=opts)
        return layer, vb.TsdfIntegratorFactory.create(kind, cfg, layer)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    # page-locked host clouds from the engine's own allocator (vbx_host_alloc = cudaHostAlloc, portable): on
    # this box it feeds the copy engine at ~50 GB/s, torch's pin_memory() pool at ~21 GB/s (scripts/e2e_probe.py)
    host_alloc_layer, _ = fresh(0, 1)
    hx, hc = [], []
    for s_ in scans:
        a = host_alloc_layer.hostBuffer(s_[0].shape, np.float32)
        b = host_alloc_layer.hostBuffer(s_[1].shape, np.uint8)
        a[...] = s_[0]
        b[...] = s_[1]
        hx.append(a)
        hc.append(b)
    d_xyz = [torch.from_numpy(s[0]).to(dev) for s in scans]
    d_rgba = [torch.from_numpy(s[1]).to(dev) for s in scans]
    pts_timed = float(sum(npts[args.warmup:]))
    steps = max(1, args.steps)

    # ---- (1a) the synchronous call: returns when the scan is in the map (one host round trip per scan)
    layer, integ = fresh()
    esdf_int = None
    if do_esdf:
        esdf_layer = vb.Layer(conf["voxel"], 16, voxel_type="esdf")
        esdf_int = vb.EsdfIntegrator(vb.EsdfIntegratorConfig(max_distance_m=2.0, default_distance_m=2.0,
                                                              min_distance_m=conf["cfg"]["default_truncation_distance"] / 2,
                                                              min_diff_m=1e-3), layer, esdf_layer)

    def sync_step(i):
        integ.integratePointCloudDevice((scans[i][2], scans[i][3]), d_xyz[i].data_ptr(), d_rgba[i].data_ptr(), npts[i])
        if esdf_int is not None:
            esdf_int.updateFromTsdfLayer(True)

    for i in range(args.warmup):
        sync_step(i)
    barrier()
    layer.timerStart()
    U = B = K = 0
    for i in range(args.warmup, n_total):
        sync_step(i)
        c = integ.counters()
        U += c["voxels_touched"]
        B += c["blocks_touched"]
        K += c["updates"]
    sync_ms = layer.timerStopMs()
    barrier()
    if do_esdf and args.dump_outputs and rank == 0:  # with the ESDF update after every scan this is the timed path
        dump_outputs(args.dump_outputs, layer, esdf_layer)
    del layer, integ, esdf_int
    # ---- (1b) headline: the same K scans submitted back to back (vbx_tsdf_integrate_async): stages of
    # neighbouring scans overlap; timed on the device until the last scan is in the map.  With the ESDF
    # update after every scan (C4) the calls are synchronous by nature: (1a) is the number.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if do_esdf:
        dev_ms, wall_ms, launches, last_counters, n_blocks = sync_ms, sync_ms, 0, {}, 0
        sampler.mark_begin()
        time.sleep(0.05)
        sampler.mark_end()
    else:
        layer, integ = fresh()
        for i in range(args.warmup):
            integ.integratePointCloudAsync((scans[i][2], scans[i][3]), d_xyz[i].data_ptr(), d_rgba[i].data_ptr(), npts[i])
        layer.sync()
        barrier()
        launches_before = integ.counters()["kernel_launches_total"]
        sampler.mark_begin()
        layer.timerStart()
        t0 = time.perf_counter()
        for i in range(args.warmup, n_total):
            integ.integratePointCloudAsync((scans[i][2], scans[i][3]), d_xyz[i].data_ptr(), d_rgba[i].data_ptr(), npts[i])
        dev_ms = layer.timerStopMs()  # drains the pipeline first
        sampler.mark_end()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        last_counters = integ.counters()
        launches = last_counters["kernel_launches_total"] - launches_before
        n_blocks = layer.getNumberOfAllocatedBlocks()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, layer)
    clocks = sampler.stop() if rank == 0 else None
    dev_ms, wall_ms, sync_ms = reduce_max(dev_ms, wall_ms, sync_ms)
    value = pts_timed / (dev_ms * 1e-3)

    # ---- (2) e2e: the reference-facing call with HOST buffers, H2D inside the timed region ----
    layer2, integ2 = fresh()
    esdf2 = None
    if do_esdf:
        esdf2_layer = vb.Layer(conf["voxel"], 16, voxel_type="esdf")
        esdf2 = vb.EsdfIntegrator(vb.EsdfIntegratorConfig(max_distance_m=2.0, default_distance_m=2.0,
                                                           min_distance_m=conf["cfg"]["default_truncation_distance"] / 2,
                                                           min_diff_m=1e-3), layer2, esdf2_layer)

    def e2e_sync_step(i):
        integ2.integratePointCloud((scans[i][2], scans[i][3]), hx[i], hc[i])
        if esdf2 is not None:
            esdf2.updateFromTsdfLayer(True)
        return integ2.counters()  # the step's result block (counters) read back on the host

    for i in range(args.warmup):
        e2e_sync_step(i)
    barrier()
    layer2.timerStart()
    for i in range(args.warmup, n_total):
        e2e_sync_step(i)
    e2e_sync_ms = layer2.timerStopMs()
    barrier()
    if do_esdf:
        # the ESDF update after every scan makes the calls synchronous by nature
        e2e_ms = e2e_pageable_ms = e2e_sync_ms
    else:
        del layer2, integ2
        # headline e2e: host (page-locked) clouds submitted back to back; every step's H2D copy and the
        # D2H read of its result block (256 B of counters / status) are inside the pipeline
        layer2, integ2 = fresh()
        for i in range(args.warmup):
            integ2.integratePointCloudAsync((scans[i][2], scans[i][3]), hx[i], hc[i])
        layer2.sync()
        barrier()
        layer2.timerStart()
        for i in range(args.warmup, n_total):
            integ2.integratePointCloudAsync((scans[i][2], scans[i][3]), hx[i], hc[i])
        e2e_ms = layer2.timerStopMs()
        barrier()
        # ... and from ordinary pageable memory (what an unmodified caller's Pointcloud is)
        layer2b, integ2b = fresh()
        for i in range(args.warmup):
            integ2b.integratePointCloudAsync((scans[i][2], scans[i][3]), scans[i][0], scans[i][1])
        layer2b.sync()
        barrier()
        layer2b.timerStart()
        for i in range(args.warmup, n_total):
            integ2b.integratePointCloudAsync((scans[i][2], scans[i][3]), scans[i][0], scans[i][1])
        e2e_pageable_ms = layer2b.timerStopMs()
        barrier()
        del layer2b, integ2b
    e2e_ms, e2e_sync_ms, e2e_pageable_ms = reduce_max(e2e_ms, e2e_sync_ms, e2e_pageable_ms)
    e2e_value = pts_timed / (e2e_ms * 1e-3)
    h2d = int(np.mean([16 * n for n in npts[args.warmup:]]))

    # ---- N > 1: the union of the shards must be the single-GPU map; cost of read replicas -------
    shard_info = None
    if world > 1:
        import hashlib

        sl = sharded.ShardedLayer(layer2)
        gathered = sl.gather()
        t0 = time.perf_counter()
        n_recv = sl.sync_replicas()
        torch.cuda.synchronize()
        sync_replica_ms = (time.perf_counter() - t0) * 1e3
        if rank == 0:
            ls, isg = fresh(0, 1)
            for i in range(n_total):
                isg.integratePointCloud((scans[i][2], scans[i][3]), hx[i], hc[i])
            single = ls.blocks()

            def dig(b):
                hsh = hashlib.sha256()
                for k in sorted(b):
                    hsh.update(np.asarray(k, np.int32).tobytes())
                    hsh.update(b[k].tobytes())
                return hsh.hexdigest()[:16]

            shard_info = {"union_of_shards_digest": dig(gathered), "single_gpu_digest": dig(single),
                          "union_equals_single_gpu_map": dig(gathered) == dig(single), "blocks": len(single),
                          "blocks_owned_by_rank0": int(sum(1 for k in gathered if sharded.block_owner([k], world)[0] == 0)),
                          "sync_replicas_all_blocks_wall_ms": sync_replica_ms, "blocks_received_rank0": n_recv}
            del ls, isg
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- (3) per-stage device time (profiling pass), roofline ---------------------------------
    layer3, integ3 = fresh(0, 1)
    for i in range(n_total):
        if i == args.warmup:
            layer3.setStageProfiling(True)
        integ3.integratePointCloudDevice((scans[i][2], scans[i][3]), d_xyz[i].data_ptr(), d_rgba[i].data_ptr(), npts[i])
    stages = {k: v for k, v in layer3.stageMs().items() if v[1] > 0}
    del layer3, integ3
    n_mean, u_mean, b_mean, k_mean = pts_timed / steps, U / steps, B / steps, K / steps
    # SURVEY.md section 8(d): algorithmic bytes per scan = 16 N + 24 U + 20 B; each stage owns the part of
    # it that it must move (the cloud is algorithmically read once: by the stages up to the bundle fold;
    # block keys / slab pointers by the ray walk; the touched voxels by the apply).  Update records, sort
    # traffic and the per-ray tables are this design's own overhead and count for nothing here.
    alg = {"point_keys": 12 * n_mean, "bundle_merge": 16 * n_mean, "ray_emit": 20 * b_mean, "apply": 24 * u_mean,
           "point_sort": 0.0, "bundle_order": 0.0, "scan": 0.0, "update_sort": 0.0, "assign": 0.0, "ray_count": 0.0}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    scan_alg = 16 * n_mean + 24 * u_mean + 20 * b_mean
    if args.traffic and world == 1:
        traffic = measure_traffic(args.config, cache_control="none")
        traffic_cold = measure_traffic(args.config, cache_control="all")
    else:
        traffic = traffic_cold = {"unavailable": "--no-traffic or N > 1"}
    top = max(stages, key=lambda k: stages[k][0]) if stages else None
    top_ms = stages[top][0] / stages[top][1] if top else None
    dom = None
    if top:
        t_bytes = None
        if "per_kernel" in traffic:
            t_bytes = sum(v["dram_bytes_per_scan"] for k, v in traffic["per_kernel"].items()
                          if k in STAGE_OF_KERNEL.get(top, ()))
        dom = {"stage": top, "kernels": list(STAGE_OF_KERNEL.get(top, ())), "avg_ms": top_ms,
               "alg_bytes_per_launch": alg.get(top, 0.0),
               "achieved": alg.get(top, 0.0) / (top_ms * 1e-3) / 1e9, "frac": alg.get(top, 0.0) / (top_ms * 1e-3) / 1e9 / peak,
               "traffic": t_bytes}
    ms_per_step = dev_ms / steps
    roofline = {"bound": "hbm", "unit": "GB/s", "peak": peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if peaks else "fallback 6650",
                # headline: SURVEY 8(d)'s whole-scan bytes over the measured time per scan
                "alg_bytes_per_launch": scan_alg, "alg_bytes_formula": "16*N + 24*U + 20*B (SURVEY.md 8d)",
                "achieved": scan_alg / (ms_per_step * 1e-3) / 1e9, "frac": scan_alg / (ms_per_step * 1e-3) / 1e9 / peak,
                # DRAM bytes per scan, all kernels of the scan: caches as the run leaves them / flushed per kernel
                "traffic": traffic.get("total_dram_bytes_per_scan"), "traffic_detail": traffic,
                "traffic_cold_cache": traffic_cold.get("total_dram_bytes_per_scan"), "traffic_cold_cache_detail": traffic_cold,
                "synchronous_call_frac": scan_alg / (sync_ms / steps * 1e-3) / 1e9 / peak,
                "dominant_kernel": dom,
                "stage_ms_per_scan": {k: round(v[0] / steps, 5) for k, v in stages.items()},
                "why_small": "a scan moves ~5 MB (1 us at HBM speed); every stage is a latency chain "
                             "(dependent loads, ordered per-voxel update chains), not a bandwidth stream"}

    # ---- (4) CPU baseline on this box's host cores, bounded sample ------------------------
    from oracle import pyoracle as po

    sample = scans[:min(len(scans), 12 if conf["scan"] != "c5_lidar_scan" else 5)]
    if world > 1:
        # (N > 1: the other ranks' GPUs idle while rank 0 measures the CPU: one thread, as calibrated at N = 1)
        sample = sample[:6]
        threads, detail = 1, {"1": "not calibrated at N > 1"}
    else:
        threads, detail = calibrate_threads(conf, sample[:3])
    which, secs = time_reference(conf, sample, threads, esdf=do_esdf)
    cpu_pts = sum(int(s[0].shape[0]) for s in sample[2:])
    cpu_value = cpu_pts / float(sum(secs[2:]))
    cpu = {"value": cpu_value, "unit": "points/s", "cores": threads, "kind": which,
           "sample": f"{len(sample) - 2} scans of the workload after 2 warm-up scans; {kind} integrator "
                     f"with integrator_threads={threads} (fastest of {detail} ms/scan; {os.cpu_count()} logical cores)"}
    try:  # the same translation units at -O3 -march=x86-64-v3 (BASELINE.md): a faster-than-stock build, for context
        if po.available("reference_o3"):
            _, secs3 = time_reference(conf, sample, threads, which="reference_o3", esdf=do_esdf)
            cpu["o3_x86_64_v3"] = {"value": cpu_pts / float(sum(secs3[2:])), "cores": threads}
    except Exception as exc:
        cpu["o3_x86_64_v3"] = {"error": repr(exc)}

    # ---- (5) parity against the reference itself (one thread) on the first scans -----------
    parity = None
    if kind != "fast":
        from tests.parity import compare_tsdf

        layer4, integ4 = fresh(0, 1)
        pw = "reference" if po.available("reference") else "port"
        omap = po.OracleMap(po.OracleLib(pw), po.TsdfConfig(integrator_threads=1, **conf["cfg"]), conf["voxel"], 16)
        for s in scans[:3]:
            integ4.integratePointCloud((s[2], s[3]), s[0], s[1])
            omap.integrate(KIND_ID[kind], s)
        rep = compare_tsdf(layer4, omap)
        parity = {"against": pw + " (integrator_threads=1)", "scans": 3, "blocks_equal": rep["blocks_equal"],
                  "max_rel_err": rep.get("max_rel_err"), "bit_exact_voxels": rep.get("n_bit_exact"),
                  "voxels": rep.get("n_voxels"), "color_mismatch": rep.get("color_mismatch")}
        del layer4, integ4

    # ---- (6) the callers either side of the path (SURVEY.md 8d C4, 8f N3): ESDF update and
    # incremental mesh after every scan; device time per call, not part of `value`
    downstream = None
    if args.config == "bench" and world == 1:
        try:
            layer5, integ5 = fresh(0, 1)
            esdf5 = vb.Layer(conf["voxel"], 16, voxel_type="esdf")
            e5 = vb.EsdfIntegrator(vb.EsdfIntegratorConfig(max_distance_m=2.0, default_distance_m=2.0,
                                                           min_distance_m=0.1, min_diff_m=1e-3), layer5, esdf5)
            mesh5 = vb.MeshLayer(layer5.block_size())
            m5 = vb.MeshIntegrator(vb.MeshIntegratorConfig(), layer5, mesh5)
            t_ms5, e_ms5, m_ms5, m_wall5 = [], [], [], []
            k5 = min(n_total, 12)
            for i in range(k5):
                integ5.integratePointCloudDevice((scans[i][2], scans[i][3]), d_xyz[i].data_ptr(), d_rgba[i].data_ptr(), npts[i])
                t_ms5.append(integ5.lastDeviceMs())
                e5.updateFromTsdfLayer(True)
                e_ms5.append(e5.lastDeviceMs())
                t0 = time.perf_counter()
                m5.generateMesh(True, True)
                m_wall5.append((time.perf_counter() - t0) * 1e3)
                m_ms5.append(m5.lastDeviceMs())
            w = slice(min(3, k5 - 1), None)
            ec = e5.counters()
            downstream = {"scans": k5, "tsdf_sync_device_ms": float(np.mean(t_ms5[w])),
                          "esdf_incremental_device_ms": float(np.mean(e_ms5[w])),
                          "mesh_incremental_device_ms": float(np.mean(m_ms5[w])),
                          "mesh_incremental_wall_ms_incl_download": float(np.mean(m_wall5[w])),
                          "mesh_vertices_last_call": int(m5.last_vertices), "mesh_blocks_last_call": int(m5.last_blocks),
                          "esdf_last_counters": ec,
                          "esdf_roofline": {"alg_bytes_formula": "(12+20+20)*4096*B_upd + 40*R (SURVEY.md 8d)",
                                            "alg_bytes": 52 * 4096 * ec.get("blocks", 0) + 40 * ec.get("relaxations", 0),
                                            "frac": (52 * 4096 * ec.get("blocks", 0) + 40 * ec.get("relaxations", 0)) /
                                                    max(1e-9, e_ms5[-1] * 1e-3) / 1e9 / peak},
                          "note": "Merged + EsdfIntegrator::updateFromTsdfLayer(true) + MeshIntegrator::generateMesh(true, true) "
                                  "after every scan (config C4 + N3)"}
        except Exception as exc:  # never lose the headline line to an optional section
            downstream = {"error": repr(exc)}

    config = config_dict(conf, scans[args.warmup:])  # (exactly the reference arm's object)
    workload_stats = {"updates_per_scan_mean": k_mean, "voxels_touched_per_scan_mean": u_mean,
                      "blocks_touched_per_scan_mean": b_mean, "map_blocks_after_run": n_blocks}
    parallelism = ("single GPU" if world == 1 else
                   f"own{world}: ONE map sharded over {world} GPUs by block ownership; every rank receives every scan, "
                   "folds and walks all rays, applies only the voxels of its own blocks; no collective while integrating")
    line = {
        "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config, "workload_stats": workload_stats, "parallelism": parallelism, "clocks": clocks,
        "wall_ms_per_step": wall_ms / steps,
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": 256 * world,
                "ms_per_step": e2e_ms / steps, "submission": "vbx_tsdf_integrate_async, page-locked host clouds (vbx_host_alloc)"
                + (" (every rank copies the whole cloud over its own PCIe link)" if world > 1 else ""),
                "synchronous_call": {"value": pts_timed / (e2e_sync_ms * 1e-3), "ms_per_step": e2e_sync_ms / steps},
                "pageable_host_memory": {"value": pts_timed / (e2e_pageable_ms * 1e-3), "ms_per_step": e2e_pageable_ms / steps}},
        "submission": "vbx_tsdf_integrate_async: scans queued back to back, timed until the last one is in the map",
        "synchronous_call": {"value": pts_timed / (sync_ms * 1e-3), "ms_per_step": sync_ms / steps,
                             "note": "vbx_tsdf_integrate_device, returns when the scan is in the map"
                             + (" + EsdfIntegrator::updateFromTsdfLayer(true)" if do_esdf else "")},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
        "last_counters": last_counters, "downstream": downstream,
    }
    if shard_info is not None:
        line["sharded_map"] = shard_info
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="bench", choices=sorted(CONFIGS))
    ap.add_argument("--trunc", type=float, default=None, help="override default_truncation_distance (C2: 4.0 = the literal '4 m')")
    ap.add_argument("--no-traffic", dest="traffic", action="store_false", help="skip the ncu DRAM-traffic pass")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the map they produced as DIR/<name>.npy (with N > 1: rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    conf = dict(CONFIGS[args.config])
    if args.trunc is not None:
        conf["cfg"] = dict(conf["cfg"], default_truncation_distance=args.trunc)
        conf["workload"] += f"_trunc{args.trunc:g}"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # Exactly ONE line goes to stdout: the JSON.  Libraries (NCCL's version banner, make) write to file
    # descriptor 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON line is
    # written to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    import __graft_entry__ as g

    if rank == 0:
        old = sys.stdout
        sys.stdout = sys.stderr
        try:
            if args.impl == "reference":
                g.build_oracle()  # the reference arm loads nothing of the engine
            else:
                g.build()
        finally:
            sys.stdout = old
    if args.traffic_child:
        traffic_child(conf)
    elif args.impl == "reference":
        run_reference_arm(args, conf, rank)
    else:
        run_ours(args, conf, rank, world)


if __name__ == "__main__":
    main()
