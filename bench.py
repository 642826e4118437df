#!/usr/bin/env python
"""bench.py -- scan-to-map ICP registrations/s on synthetic 64-beam x 1024-azimuth LiDAR clouds (BASELINE.json metric).

Workload (config[1] of BASELINE.json): the scan-to-map odometry loop with the reference's Lua defaults
(voxel 0.1 m, MinMaxRadius 2-30 m, knn 20 / 3 m, max corr. 1 m, <= 50 iterations, map voxel 0.1 m, PointToPlaneIcp,
downsampling ratio 0.3, fitness gate 0.7) in STEADY STATE: every chain first drives one full lap of the closed 59 m loop
(118 scans, untimed) so that its map holds the whole courtyard before anything is timed.

One "step" = every one of the `chains` independent odometry chains on this GPU advances by `scans_per_step` scans, each
through the whole hot path:
    S1 crop+voxel+normals+select -> S2 map-patch crop + NN index + point-to-plane ICP -> fitness gate -> F1 map fusion.
Chains are independent trajectories (one b2s handle / CUDA stream each), the units that shard across GPUs
(weak scaling, no data-path collective; SURVEY.md 8e).  Within a chain the scans stay strictly sequential.

  value : registrations/s with the raw scans already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e   : the same, every scan uploaded from pinned host memory (float32) and its RegistrationResult read back to the
          host, through the public mapper API (one C call per scan)
  chain_sweep / single_chain_latency_ms : the same resident measurement at 1, 4, 8, 16, 32 chains (N = 1 only)
  roofline     : the dominant kernel group, timed live with CUDA events on its own stream (one eager chain, steady-state map)
  config3/4/5  : the other configurations of BASELINE.json, device-timed in the same run (open3d_slam_b200/benchmarks.py)
  cpu_baseline : the CPU oracle (oracle/, "port" of the reference's Open3D path) on a bounded sample, rank 0 only
  --impl reference : the same workload on the host cores through the oracle only (no GPU code on that path)
  --dump-outputs DIR : after the timed steps, the last step's outputs as float64 DIR/<name>.npy (dump_last_step).  The inputs
          are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import copy
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (no __pycache__ either)

from open3d_slam_b200 import synth  # noqa: E402
from open3d_slam_b200 import workloads as W  # noqa: E402

METRIC = "scan-to-map ICP registrations/sec (64x1024-pt clouds)"
UNIT = "registrations/s"
WORKLOAD = "config2: scan-to-map odometry loop, synthetic 64x1024 LiDAR, voxel 0.1 m, Lua defaults, PointToPlaneIcp, steady-state map"
SCAN_SETS = 8   # noise realisations of the lap; chain c replays set c % SCAN_SETS
LAP = int(round(synth.loop_length() / 0.5))   # scans per lap of the closed loop (118)
RESULT_SLOTS = 256                # per-engine ring of RegistrationResults (b2s_scan_result_fetch)
DUMP_BYTES = 64 << 20             # --dump-outputs writes at most this much
DUMP_MAP_SAMPLE = 16384           # map points per chain in the dump (fewer when DUMP_BYTES would be exceeded)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def make_config(args):
    """The SAME dict in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "chains_per_gpu": args.chains, "scans_per_step": args.scans_per_step, "downsampling_ratio": args.ratio,
            "rays_per_scan": 65536, "pregrown_scans_per_chain": LAP,
            "l2": "256 MiB write between timed steps (outside the event brackets)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle restating the reference's own CPU path (never on the product path)
# ----------------------------------------------------------------------------------------------------------------------
class OracleChain:
    def __init__(self, ratio, seed):
        from oracle import oracle as O
        self.O = O
        self.wide = O.cropper("MinMaxRadius", 2.0, 30.0)
        self.narrow = O.cropper("MinMaxRadius", 2.0, 30.0)
        self.ratio, self.seed = ratio, seed
        self.map_x = np.zeros((0, 3)); self.map_n = np.zeros((0, 3)); self.pose = np.eye(4)
        self.first = True

    def step(self, raw32, delta):
        O = self.O
        (mx, mn), (ax, an) = O.process_scan(raw32.astype(np.float64), self.wide, self.narrow, 0.1, 20, 3.0, self.ratio, self.seed)
        if self.first:
            self.map_x, self.map_n = O.submap_insert_scan(self.map_x, self.map_n, mx, mn, np.eye(4), 0.1, self.wide)
            self.first = False
            return None
        c = O.cropper("MinMaxRadius", 2.0, 30.0, center=self.pose[:3, 3])
        px, pn = O.crop(c, self.map_x, self.map_n)
        res = O.registration_icp_p2plane(ax, px, pn, 1.0, self.pose @ delta, max_iter=50)
        if res.fitness >= 0.7:
            self.pose = res.T
            self.map_x, self.map_n = O.submap_insert_scan(self.map_x, self.map_n, mx, mn, self.pose, 0.1, self.wide)
        return res


def run_reference_arm(args):
    """The reference's CPU path (oracle port) on the same workload: `chains` chains in parallel, each pre-grown over one lap, then W + K
    steps; a step here is a BOUNDED SAMPLE of the GPU arm's step -- one of its `scans_per_step` scans per chain."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import oracle as O
    from concurrent.futures import ThreadPoolExecutor
    cores = os.cpu_count() or 1
    chains = args.chains
    lp = W.ClosedLoop()
    per = max(1, cores // chains)
    os.environ["OMP_NUM_THREADS"] = str(per)
    O.lib()
    cs = [OracleChain(args.ratio, 3) for _ in range(chains)]
    pool = ThreadPoolExecutor(max_workers=chains)
    scans = {}

    def scan(c, k):
        key = (c % SCAN_SETS, k % lp.L)
        if key not in scans:
            scans[key] = lp.scan(k, seed=1000 * (c % SCAN_SETS) + (k % lp.L))
        return scans[key]

    def do_step(k):
        list(pool.map(lambda c: cs[c].step(scan(c, k), lp.delta(k)), range(chains)))

    t_grow = time.perf_counter()
    for k in range(lp.L):          # untimed: steady-state map
        do_step(k)
    t_grow = time.perf_counter() - t_grow
    k = lp.L
    for _ in range(args.warmup):
        do_step(k); k += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        do_step(k); k += 1
    dt = time.perf_counter() - t0
    value = chains * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": make_config(args),
            "observed": {"map_points": int(np.mean([len(c.map_x) for c in cs])), "pregrow_s": t_grow},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{chains} chains x {args.steps} scans on steady-state maps (one of the {args.scans_per_step} scans of every GPU-arm step), "
                                       f"{chains} chains in parallel x {per} OpenMP threads"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(lp, ratio, n_sample):
    from oracle import oracle as O
    O.lib()
    ch = OracleChain(ratio, 3)
    for k in range(lp.L):          # steady-state map first (untimed)
        ch.step(lp.scan(k, seed=k % lp.L), lp.delta(k))
    t0 = time.perf_counter()
    for k in range(lp.L, lp.L + n_sample):
        ch.step(lp.scan(k, seed=k % lp.L), lp.delta(k))
    dt = time.perf_counter() - t0
    return {"value": n_sample / dt, "unit": UNIT, "cores": O.num_threads(), "kind": "port", "map_points": int(len(ch.map_x)),
            "sample": f"1 chain x {n_sample} consecutive scans on its steady-state map (crop+voxel+normals+select, KD-tree rebuild + ICP, map fusion), "
                      f"{O.num_threads()} OpenMP threads"}


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
def dump_last_step(out_dir, maps, last_slot, scans, suffix=""):
    """Writes what the timed path returned in its last step, as float64 .npy files: every chain's RegistrationResult for each of
    the step's `scans` scans (shape chains x scans ...), every chain's submap pose and size, and a seeded sample of every chain's
    map.  The map is sorted before sampling, so the sample does not depend on the order the device stores the points in."""
    res = [[m.fetchResult((last_slot[c] - scans + 1 + j) % RESULT_SLOTS) for j in range(scans)] for c, m in enumerate(maps)]
    out = {"transformation": np.array([[r.transformation_ for r in rc] for rc in res]),
           "fitness": np.array([[r.fitness_ for r in rc] for rc in res]),
           "inlier_rmse": np.array([[r.inlier_rmse_ for r in rc] for rc in res]),
           "n_corr": np.array([[r.n_corr for r in rc] for rc in res], dtype=np.float64),
           "iters": np.array([[r.iters for r in rc] for rc in res], dtype=np.float64),
           "pose": np.array([m.submap.getPose() for m in maps]),
           "map_size": np.array([m.submap.size() for m in maps], dtype=np.float64)}
    clouds = [m.submap.getMapPointCloud() for m in maps]
    budget = DUMP_BYTES - sum(a.nbytes for a in out.values())
    n_pick = min([DUMP_MAP_SAMPLE, max(0, budget) // (48 * len(maps))] + [len(x) for x, _ in clouds])
    xs, ns = [], []
    for x, n in clouds:
        order = np.lexsort((n[:, 2], n[:, 1], n[:, 0], x[:, 2], x[:, 1], x[:, 0]))
        pick = order[np.sort(np.random.default_rng(0).choice(len(x), size=n_pick, replace=False))]
        xs.append(x[pick]); ns.append(n[pick])
    out["map_xyz_sample"] = np.array(xs); out["map_normals_sample"] = np.array(ns)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_b2s_arm(args):
    import torch
    import torch.distributed as dist
    from open3d_slam_b200 import benchmarks as B
    from open3d_slam_b200 import engine as E
    from open3d_slam_b200 import _lib as L

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the b2s engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    chains, K, Wu, S = args.chains, args.steps, args.warmup, args.scans_per_step
    sweep = [] if (world > 1 or args.no_sweep) else sorted(set(int(x) for x in args.sweep.split(",") if x))
    n_chains = max([chains] + sweep)
    lp = W.ClosedLoop()
    Lp = lp.L
    sets = min(n_chains, SCAN_SETS)
    t_gen = time.perf_counter()
    scans = [[lp.scan(k, seed=1000 * s + k) for k in range(Lp)] for s in range(sets)]
    deltas = [np.ascontiguousarray(lp.delta(k)) for k in range(1, Lp + 1)]   # periodic in k with period L for k >= 1
    t_gen = time.perf_counter() - t_gen
    pts = int(np.mean([len(s) for s in scans[0]]))

    def delta(k):
        return deltas[(k - 1) % Lp]

    params = E.MapperParameters(seed=3)
    params.scanProcessing.downSamplingRatio = args.ratio
    params.nnCellSize = args.nn_cell
    main = torch.cuda.current_stream(dev)
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_chains)]
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    use_graph = not args.no_graph

    # ---------------- chains: one engine / stream / mapper each, pre-grown over one lap (untimed) ----------------
    engs = [E.Engine(params, device=local, cuda_stream=streams[c].cuda_stream) for c in range(n_chains)]
    maps = [E.Mapper(e, args.map_capacity) for e in engs]
    dev_clouds = [[engs[s].cloud(scans[s][k]) for k in range(Lp)] for s in range(sets)]   # resident inputs (set s is uploaded through engine s)
    for e in engs:
        e.synchronize()
    for c in range(n_chains):   # first scan: pre-process and insert with identity (Mapper.cpp:105-114)
        maps[c].addRangeMeasurement(dev_clouds[c % sets][0], None)
        maps[c].submap.setPose(np.eye(4))
        engs[c].synchronize()
    staging = [maps[c].enableGraph(65536) for c in range(n_chains)] if use_graph else None
    kpos = [1] * n_chains        # next scan index of every chain

    from concurrent.futures import ThreadPoolExecutor
    host_threads = args.host_threads if args.host_threads > 0 else (1 if use_graph else 8)
    pool = ThreadPoolExecutor(max_workers=host_threads) if host_threads > 1 else None

    def fan_out(fn, n):
        if pool is None:
            for c in range(n):
                fn(c)
        else:
            list(pool.map(fn, range(n)))

    slot_log = {}

    def one_resident(c):
        k = kpos[c]
        src = dev_clouds[c % sets][k % Lp]
        if staging is not None:   # device->device copy of the resident scan into the graph's staging cloud (1.3 MB)
            maps[c].stageCopy(src)
            slot_log[c] = maps[c].addRangeMeasurementAsync(staging[c], delta(k))
        else:
            slot_log[c] = maps[c].addRangeMeasurementAsync(src, delta(k), slot=k % 256)
        kpos[c] = k + 1

    def timed_region(one, n, nsteps, nscans):
        """nsteps steps of nscans scans for chains 0..n-1; every step is bracketed by events on the main stream, the chain
        streams fork/join around it, the L2 is flushed (256 MiB write) outside the brackets.  Returns per-step device ms."""
        evs = []
        for _ in range(nsteps):
            flush_buf.zero_()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(main)
            for s in streams[:n]:
                s.wait_event(a)
            for _s in range(nscans):
                fan_out(one, n)
            for s in streams[:n]:
                d = torch.cuda.Event(); d.record(s); main.wait_event(d)
            b.record(main)
            evs.append((a, b))
        torch.cuda.synchronize(dev)
        return [a.elapsed_time(b) for a, b in evs]

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    t_grow = time.perf_counter()
    timed_region(one_resident, n_chains, 1, Lp - 1)      # the rest of lap 0: maps reach steady state
    for c in range(n_chains):
        engs[c].synchronize()                            # surfaces a device status error (capacity, ...) here, not in the timed region
    t_grow = time.perf_counter() - t_grow
    map_pts0 = int(np.mean([m.submap.size() for m in maps[:chains]]))

    # ---------------- value: inputs resident in HBM ----------------
    timed_region(one_resident, chains, Wu, S)
    l0 = sum(e.launches for e in engs[:chains])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    t_wall = time.perf_counter()
    step_ms = timed_region(one_resident, chains, K, S)
    t_wall = time.perf_counter() - t_wall
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = sum(e.launches for e in engs[:chains]) - l0
    if args.dump_outputs:   # before the sweep and e2e runs below overwrite the result rings
        dump_last_step(args.dump_outputs, maps[:chains], slot_log, S, f"_rank{rank}" if world > 1 else "")
    ms_total = max_over_ranks(float(np.sum(step_ms)))
    value = world * chains * K * S / (ms_total * 1e-3)
    # the last scan of every chain: iterations, source size, sanity against ground truth
    last = [maps[c].fetchResult(slot_log[c]) for c in range(chains)]
    iters_last = np.array([r.iters for r in last]); fit_last = np.array([r.fitness_ for r in last])
    nsrc_last = np.array([r.n_corr / max(r.fitness_, 1e-12) for r in last])
    pose_err = max(float(np.linalg.norm(maps[c].submap.getPose()[:3, 3] - lp.map_frame_pose(kpos[c] - 1)[:3, 3])) for c in range(chains))
    map_pts = int(np.mean([m.submap.size() for m in maps[:chains]]))

    # ---------------- chain sweep (N = 1): same resident measurement at other chain counts ----------------
    sweep_out, latency_ms = {}, None
    if sweep:
        for n in sweep:
            timed_region(one_resident, n, 1, 8)
            sm = timed_region(one_resident, n, 4, 24)
            per_scan_step = float(np.median(sm)) / 24.0          # ms for all n chains to advance one scan
            sweep_out[str(n)] = {"registrations_per_s": n / per_scan_step * 1e3, "ms_per_scan_step": per_scan_step}
            if n == 1:
                latency_ms = per_scan_step
        sweep_out[str(chains)] = {"registrations_per_s": value, "ms_per_scan_step": ms_total / (K * S)}
    # latency mode: one chain alone with the registration spread over 16 SMs instead of 8 (b2s_config.icp_cluster_ctas; the default
    # of 8 is the throughput setting the headline is measured with -- 16-SM clusters of many concurrent chains queue behind each other)
    latency16_ms = None
    if sweep and 1 in sweep:
        p16 = copy.deepcopy(params); p16.icpClusterCtas = 16
        engs[0].set_parameters(p16)
        timed_region(one_resident, 1, 1, 8)
        latency16_ms = float(np.median(timed_region(one_resident, 1, 4, 24))) / 24.0
        engs[0].set_parameters(params)
        timed_region(one_resident, 1, 1, 4)

    # ---------------- e2e: host buffers in, results out, every scan ----------------
    pinned = [[torch.from_numpy(scans[s][k]).pin_memory() for k in range(Lp)] for s in range(sets)]
    res_sz = ctypes.sizeof(L.Result)
    RING = 256
    res_pinned = torch.zeros((chains, RING, res_sz), dtype=torch.uint8).pin_memory()   # every scan's RegistrationResult lands here
    h2d = chains * S * pts * 12
    d2h = chains * S * res_sz
    e2e_last = {}

    def one_e2e(c):
        k = kpos[c]
        t = pinned[c % sets][k % Lp]   # one C call enqueues: H2D of the float32 scan, the whole chain, D2H of the RegistrationResult
        maps[c].addRangeMeasurementHostAsync(t.data_ptr(), t.shape[0], delta(k), res_pinned[c, k % RING].data_ptr())
        e2e_last[c] = k % RING
        kpos[c] = k + 1

    timed_region(one_e2e, chains, Wu, S)
    barrier()
    e2e_ms = timed_region(one_e2e, chains, K, S)
    barrier()
    ms_e2e = max_over_ranks(float(np.sum(e2e_ms)))
    e2e_value = world * chains * K * S / (ms_e2e * 1e-3)
    e2e_res = [L.Result.from_buffer_copy(res_pinned[c, e2e_last[c]].numpy().tobytes()) for c in range(chains)]
    e2e_fit = float(min(r.fitness for r in e2e_res))
    e2e_err = max(float(np.linalg.norm(np.array(r.T).reshape(4, 4)[:3, 3] - lp.map_frame_pose(kpos[c] - 1)[:3, 3])) for c, r in enumerate(e2e_res))

    # ---------------- per-kernel-group device times: one eager chain on a copy of chain 0's steady-state map ----------------
    mx, mn = maps[0].submap.getMapPointCloud()
    pose0 = maps[0].submap.getPose()
    k0 = kpos[0]
    p_eng = E.Engine(params, device=local, cuda_stream=streams[0].cuda_stream)
    p_map = E.Mapper(p_eng, args.map_capacity)
    p_map._first = False
    p_map.submap.setMapPointCloud(p_eng.cloud(mx, mn))
    p_map.submap.setPose(pose0)
    kp = 10
    for j in range(3):
        p_map.addRangeMeasurementAsync(dev_clouds[0][(k0 + j) % Lp], delta(k0 + j), slot=j)
    p_eng.synchronize()
    p_eng.profile_enable(True)
    p_eng.profile_read()
    lp0 = p_eng.launches
    for j in range(3, 3 + kp):
        flush_buf.zero_()
        torch.cuda.synchronize(dev)
        p_map.addRangeMeasurementAsync(dev_clouds[0][(k0 + j) % Lp], delta(k0 + j), slot=j)
    prof = p_eng.profile_read()
    launches_per_scan_eager = (p_eng.launches - lp0) / kp
    p_eng.profile_enable(False)
    p_res = [p_map.fetchResult(j) for j in range(3, 3 + kp)]
    p_iters = np.array([r.iters for r in p_res]); p_nsrc = np.array([r.n_corr / max(r.fitness_, 1e-12) for r in p_res])
    p_map.submap.free()
    p_eng.close()

    # ---------------- roofline of the dominant kernel group (live CUDA events on its stream) ----------------
    peak, peak_src = B.hbm_peak()
    kinds = {k: v for k, v in prof.items() if v[1] > 0}
    dom = max(kinds, key=lambda k: kinds[k][0]) if kinds else "icp"
    bytes_icp = float(np.mean(72.0 * p_nsrc * (p_iters + 1)))      # algorithmic bytes per launch, fp64 layout (DESIGN.md section 5)
    m_vox = float(np.mean(p_nsrc)) / max(args.ratio, 1e-9)         # points entering normal estimation (before the ratio down-sample)
    bytes_by_kind = {"icp": bytes_icp, "normals": 24.0 * float(np.mean(p_nsrc)) * (20 + 2), "voxel": 24.0 * pts + 24.0 * m_vox}
    dom_for_roof = dom if dom in bytes_by_kind else "icp"
    ab = bytes_by_kind[dom_for_roof]
    dur_ms = prof[dom_for_roof][0] / max(prof[dom_for_roof][1], 1)
    achieved = ab / (dur_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None   # DRAM bytes per launch of that kernel from the committed ncu --set full capture
    for tp in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tpath):
            ent = json.load(open(tpath)).get(dom_for_roof)
            if ent:
                traffic, traffic_src = ent["bytes_per_launch"], ent["source"]
                break
    roofline = {"bound": "hbm", "kernel": dom_for_roof, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "bytes_per_launch": ab, "avg_launch_ms": dur_ms,
                "note": "latency-bound: a single registration's working set is L2-resident and its iterations are sequential (SURVEY.md 8d); "
                        "the streaming kernels' fractions are under config3, the batched ICP's under config4"}
    profile = {k: {"ms_per_scan": v[0] / kp, "launch_groups_per_scan": v[1] / kp} for k, v in prof.items()}

    # ---------------- free the chains, then the other configs ----------------
    for lst in dev_clouds:
        for c_ in lst:
            c_.free()
    for m in maps:
        m.submap.free()
    for e in engs:
        e.close()
    del pinned, res_pinned
    extras = {}
    if not args.no_extras:
        xs = torch.cuda.Stream(device=dev)
        # a failure in one of the extra configurations must not cost the headline line: it is reported in place of the numbers
        # (collectives inside: every rank takes the same path unless its own run raises, which then surfaces as a hang-free error
        # because the ranks only meet again at the barriers below)
        if rank == 0:
            try:
                extras["config3"] = B.run_config3(dev, xs)
            except Exception as ex:   # noqa: BLE001
                extras["config3"] = {"error": repr(ex)}
        barrier()
        try:
            extras["config4"] = B.run_config4(dev, xs, world, rank, lp)
        except Exception as ex:   # noqa: BLE001
            if world > 1:
                raise
            extras["config4"] = {"error": repr(ex)}
        barrier()
        try:
            c5 = B.run_config5(dev, xs, world, rank, lp)
            v5 = max_over_ranks(1.0 / c5["scans_per_s_per_robot"])
            c5["scans_per_s"] = world / v5
            extras["config5"] = c5
        except Exception as ex:   # noqa: BLE001
            if world > 1:
                raise
            extras["config5"] = {"error": repr(ex)}

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_sample(lp, args.ratio, args.cpu_sample)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": make_config(args),
                "observed": {"global_chains": world * chains, "points_per_scan": pts, "map_points": map_pts, "map_points_before_timing": map_pts0,
                             "mean_icp_iters_last_scan": float(iters_last.mean()), "mean_source_points": float(nsrc_last.mean()),
                             "min_fitness_last_scan": float(fit_last.min()), "final_pose_err_m": pose_err,
                             "timed_region_s": ms_total * 1e-3, "timed_region_wall_s": t_wall, "step_ms_min_median_max": [float(np.min(step_ms)), float(np.median(step_ms)), float(np.max(step_ms))],
                             "pregrow_s": t_grow, "input_generation_s": t_gen, "launches_per_scan_graph": launches / max(chains * K * S, 1),
                             "launches_per_scan_eager": launches_per_scan_eager, "parallelism": f"{world}x{chains} independent chains"},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K,
                        "min_fitness_last_scan": e2e_fit, "final_pose_err_m": e2e_err},
                "gpu_launches": int(launches),
                "single_chain_latency_ms": latency_ms, "single_chain_latency_ms_16sm": latency16_ms, "chain_sweep": sweep_out or None,
                "roofline": roofline, "profile_chain0": profile, "cpu_baseline": cpu}
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2s", choices=["b2s", "reference"])
    ap.add_argument("--chains", type=int, default=16, help="independent odometry chains per GPU")
    ap.add_argument("--scans-per-step", type=int, default=64, help="scans every chain advances per step (timed region = steps x this)")
    ap.add_argument("--ratio", type=float, default=0.3, help="scan_processing.downsampling_ratio (Lua default 0.3)")
    ap.add_argument("--cpu-sample", type=int, default=12, help="scans in the bounded cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config3 / config4 / config5 runs")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--sweep", default="1,4,8,32", help="other chain counts measured at N = 1")
    ap.add_argument("--map-capacity", type=int, default=760_000, help="points a chain's submap can hold")
    ap.add_argument("--host-threads", type=int, default=0, help="host threads issuing the chains' launches (0 = auto: 1 with graph replay, 8 eager)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying one CUDA graph per scan")
    ap.add_argument("--nn-cell", type=float, default=0.0, help="NN grid cell edge in metres (0 = max_corr_dist / 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's registration results, poses and a map sample to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b2s":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl b2s)")
    if args.dump_outputs and args.scans_per_step > RESULT_SLOTS:
        ap.error(f"--dump-outputs keeps the last {RESULT_SLOTS} results per chain: --scans-per-step must not exceed that")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b2s_arm(args)


if __name__ == "__main__":
    main()
