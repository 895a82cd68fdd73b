#!/usr/bin/env python
"""bench.py — registrations/sec of the scan-matching hot path on B200 (BASELINE.json metric).

Default workload = BASELINE.json configs[1]: GICP odometry over a synthetic VLP-16 sequence (65 536 pts/scan,
fast_gicp defaults of the reference's launch file: k=20, max_corr 2.5 m, eps 0.01, <=64 LM iterations; keyframe rule of
apps/scan_matching_odometry_nodelet.cpp:241-252 with hdl_graph_slam.launch's keyframe_delta_trans=1.0).  One "step" is one
frame of the chain: setInputSource (upload, search grid, k-NN covariances) -> align(guess = previous motion) -> keyframe
switch, through the C ABI's b2r_odometry_matching.  The chain is sequential (frame k's guess is frame k-1's result), so at
N GPUs every rank runs an independent replica on its own slice of the sequence ("replicas only", weak scaling, no data-path
collective; the only collective is the MAX over ranks of the device time).

  value : frames already resident in HBM when the timed region starts (b2r_odometry_matching_device)
  e2e   : the same K frames from pinned HOST buffers, H2D inside the timed region, pose read back every step
  --impl reference : the CPU oracle (restatement of fast_gicp, oracle/) on the host cores, same frames, same unit

At N > 1 the default workload is BASELINE configs[3], the loop-closure candidate batch (the path that SHARDS: groups of candidates
dealt to ranks, batched device-resident registration on each GPU, one in-library ncclAllGather of 80-byte records) — the odometry
chain only replicates.  The N = 1 line carries that workload's 1-GPU figure under "loop_batch_n1" so the 1 -> N curve has its anchor,
and the strict call-by-call odometry figure (no announced next frame: what the pcl::Registration adapter can issue) under
config.strict_chain_value.

Other workloads: --workload ndt_odometry_hdl32e_128k (configs[2]), --workload loop_batch (configs[3]), --workload gicp_odometry_vlp16_64k,
--workload voxelgrid (SURVEY §8 row a5 alone), --workload kitti_pipeline (configs[4]'s per-scan chain: prefilter -> odometry in HBM); the last
two live in bench_workloads.py.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "gicp_odometry_vlp16_64k": dict(sensor="vlp16", method="FAST_GICP", params={}, config_index=1),
    "ndt_odometry_hdl32e_128k": dict(sensor="hdl32e", method="NDT_OMP", params={"reg_resolution": 1.0}, config_index=2),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 200; loop_batch: 5 passes of the whole batch)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS) + ["loop_batch", "voxelgrid", "kitti_pipeline"],
                    help="default: gicp_odometry_vlp16_64k at 1 GPU, loop_batch (the sharded path) at N > 1")
    ap.add_argument("--cpu-sample", type=int, default=6, help="frames of the same workload timed on the CPU oracle (cpu_baseline)")
    ap.add_argument("--pairs", type=int, default=256, help="loop_batch: candidate pairs per GPU")
    ap.add_argument("--fitness-max-range", type=float, default=2.5, help="loop_batch: fitness_score_max_range (hdl_graph_slam_400/kitti.launch)")
    ap.add_argument("--ref-pairs", type=int, default=16, help="--impl reference on loop_batch: candidate pairs per step on the CPU oracle")
    ap.add_argument("--distinct-shards", action="store_true", help="loop_batch at N > 1: every rank gets different keyframe groups (default: identical shards)")
    ap.add_argument("--no-anchor", action="store_true", help="N = 1 odometry line: skip the loop_batch_n1 / strict-chain extras")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="strict call-by-call chain: do not announce the next frame (no software pipelining)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="odometry workloads: after the timed steps, write what the last timed step returned as DIR/<name>.npy")
    return ap.parse_args()


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture (profiles/), or None"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:  # noqa: BLE001
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons under the benchmark's load.  nvidia-smi needs ~0.1-0.3 s to deliver its first sample and the
    default timed region is shorter than that (20 steps of 0.4 ms), so the caller (1) starts the sampler, (2) calls begin() when the timed
    region starts, (3) after the timed region keeps issuing UNTIMED steps of the same workload until `hold_needed()` says enough wall time
    has passed under load, (4) stop() keeps the samples whose timestamps lie between begin() and the end of the hold.  The metric is
    never taken from the hold steps; `window` in the result says how long the sampled window was and how many extra steps it held."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    MIN_WINDOW_S = 0.7

    def __init__(self, dev):
        self.dev, self.p, self.path = dev, None, f"/tmp/b2r_clocks_{os.getpid()}.csv"
        self.t0 = self.t1 = None
        self.extra_steps = 0

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.dev)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.p = None
        self.begin()

    def begin(self):
        self.t0 = time.time()

    def hold_needed(self):
        """True while the window under load is still too short for nvidia-smi to have sampled it"""
        return self.p is not None and self.t0 is not None and (time.time() - self.t0) < self.MIN_WINDOW_S

    def hold(self, body, sync, max_steps=100000):
        """body(k): one more untimed step of the same workload; sync(): drain the device"""
        k = 0
        while self.hold_needed() and k < max_steps:
            body(k)
            k += 1
            if (k & 15) == 0:
                sync()
        sync()
        self.extra_steps += k

    @staticmethod
    def _ts(txt):
        import datetime
        try:
            return datetime.datetime.strptime(txt.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except Exception:  # noqa: BLE001
            return None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.t1 = time.time()
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            ts = self._ts(c[0])
            if ts is not None and self.t0 is not None and not (self.t0 - 0.02 <= ts <= self.t1 + 0.02):
                continue  # taken before the timed region started
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm),
                "window": f"{self.t1 - self.t0:.2f} s under load = the timed region + {self.extra_steps} untimed steps of the same workload "
                          "(nvidia-smi delivers a sample every 50 ms after a ~0.2 s start-up; the timed region alone can be shorter than that)"}


def host_threads():
    """all host threads this process may use (torchrun exports OMP_NUM_THREADS=1: the oracle is told explicitly)"""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def best_thread_count(orc, frames, method, params):
    """The oracle is memory/latency bound and some boxes expose SMT siblings: time FIVE frames of the chain at all / half / quarter /
    eighth of the host threads (after an untimed warm-up frame each) and keep the fastest, so the CPU arm is neither handicapped by
    oversubscription nor decided by one noisy frame.  Returns (threads, {threads: frames/s})."""
    allt = host_threads()
    cands = sorted({max(1, allt // d) for d in (1, 2, 4, 8)}, reverse=True)
    sample = frames[:7]
    table = {}
    for t in cands:
        tt = oracle_odometry(orc, sample, method, params, t)[2:]  # frame 0 = keyframe, frame 1 = warm-up
        table[t] = len(tt) / sum(tt)
    best = max(table, key=lambda k: table[k])
    return best, {str(k): round(v, 2) for k, v in table.items()}


def single_thread_figure(orc, frames, method, params):
    """SURVEY 8(d): the CPU figure on ONE thread as well (one registration of the same sequence); None if it cannot be taken"""
    try:
        tt = oracle_odometry(orc, frames[:2], method, params, 1)[1:]
        return len(tt) / sum(tt)
    except Exception:  # noqa: BLE001
        return None


def make_frames(sensor, first, count, stride=8):
    from hdl_graph_slam_b200 import synth
    return [synth.scan(sensor, frame=first + k, stride=stride) for k in range(count)]


# ------------------------------------------------------------------------------------------------ reference arm (CPU oracle)
def oracle_odometry(orc, frames, method, params, threads=0):
    """The reference's per-frame work restated with the oracle: setInputSource (kd-tree + covariances) -> align -> keyframe switch.
    The target's kd-tree / covariances (GICP) or voxel map (NDT) are kept for as long as the keyframe stays, as fast_gicp / ndt_omp do."""
    kf, prev = None, np.eye(4, dtype=np.float32)
    ndt_map = None
    times = []
    for cloud in frames:
        t0 = time.perf_counter()
        if method == "FAST_GICP":
            if kf is None:
                kf = orc.GicpTarget(cloud, 20, threads)
            else:
                cov = orc.gicp_covariances(cloud, 20, threads)  # setInputSource: source kd-tree + covariances
                r = kf.align(cloud, prev, threads=threads, src_cov=cov)
                T = r["T"]
                prev = T
                if np.linalg.norm(T[:3, 3]) > 1.0:
                    kf, prev = orc.GicpTarget(cloud, 20, threads), np.eye(4, dtype=np.float32)  # setInputTarget(keyframe): kd-tree + covariances again
        else:
            if kf is None:
                kf = cloud
                ndt_map = orc.NdtMap(kf, params.get("reg_resolution", 1.0))
            else:
                r = ndt_map.align(cloud, prev, threads=threads, fixed_iterations=params.get("fixed_iterations", 30))
                T = r["T"]
                prev = T
                if np.linalg.norm(T[:3, 3]) > 1.0:
                    kf, prev = cloud, np.eye(4, dtype=np.float32)
                    ndt_map = orc.NdtMap(kf, params.get("reg_resolution", 1.0))
        times.append(time.perf_counter() - t0)
    return times


def oracle_loop_pairs(orc, groups, guesses, group_first, g_list, threads, max_range):
    """LoopDetector::matching restated with the oracle for the groups in g_list: setInputTarget once per group, then per candidate
    setInputSource (kd-tree + covariances) + align + getFitnessScore(max_range).  Returns seconds per group."""
    from hdl_graph_slam_b200 import synth
    times = []
    for g in g_list:
        tf, sfs = groups[g]
        tcloud = synth.scan("vlp16", frame=tf, stride=8)
        clouds = [synth.scan("vlp16", frame=sf, stride=8) for sf in sfs]
        t0 = time.perf_counter()
        tgt = orc.GicpTarget(tcloud, 20, threads)
        for c, cloud in enumerate(clouds):
            cov = orc.gicp_covariances(cloud, 20, threads)
            r = tgt.align(cloud, guesses[group_first[g] + c], threads=threads, src_cov=cov)
            tgt.fitness(cloud, r["T"], max_range, threads)
        times.append(time.perf_counter() - t0)
    return times


def loop_thread_count(orc, groups, guesses, group_first, max_range):
    allt = host_threads()
    table = {}
    for t in sorted({max(1, allt // d) for d in (1, 2, 4, 8)}, reverse=True):
        tt = oracle_loop_pairs(orc, groups, guesses, group_first, [0], t, max_range)
        table[t] = 8.0 / sum(tt)
    best = max(table, key=lambda k: table[k])
    return best, {str(k): round(v, 2) for k, v in table.items()}


def cpu_baseline_loop(groups, guesses, group_first, max_range, sample_groups=3):
    """cpu_baseline object of the loop-batch line: the oracle on a bounded sample (a thread sweep on group 0, then `sample_groups` groups)"""
    from oracle import oracle as orc
    orc.build()
    cores, table = loop_thread_count(orc, groups, guesses, group_first, max_range)
    g_list = [(1 + i) % len(groups) for i in range(sample_groups)]
    tt = oracle_loop_pairs(orc, groups, guesses, group_first, g_list, cores, max_range)
    n_pairs = sum(group_first[g + 1] - group_first[g] for g in g_list)
    return {"value": n_pairs / sum(tt), "unit": "registrations/s", "cores": cores, "host_threads_available": host_threads(), "thread_sweep_pairs_per_s": table,
            "kind": "port",
            "sample": f"{n_pairs} candidate pairs ({len(g_list)} keyframe groups) of the same workload: per group one kept target (kd-tree + covariances), per candidate "
                      f"source kd-tree + covariances + align + getFitnessScore, as LoopDetector::matching does; oracle = from-scratch OpenMP restatement of fast_gicp"}


def run_reference_loop(args, rank):
    """--impl reference on the loop-closure batch: the CPU oracle on a bounded sample of the same candidate pairs per step"""
    if rank != 0:
        return
    from oracle import oracle as orc
    from hdl_graph_slam_b200 import batch
    orc.build()
    n_groups = max(1, args.pairs // batch.GROUP) * max(1, args.gpus)
    groups, guesses, group_first = batch.loop_workload(n_groups, "vlp16")
    gps = max(1, args.ref_pairs // batch.GROUP)  # groups per step
    cores, table = loop_thread_count(orc, groups, guesses, group_first, args.fitness_max_range)
    steps = min(args.steps, 40)  # bounded: at most 40 steps x ref_pairs pairs
    g_list = [(1 + i) % n_groups for i in range((steps + args.warmup) * gps)]
    oracle_loop_pairs(orc, groups, guesses, group_first, g_list[: args.warmup * gps], cores, args.fitness_max_range)
    tt = oracle_loop_pairs(orc, groups, guesses, group_first, g_list[args.warmup * gps:], cores, args.fitness_max_range)
    n_pairs = len(tt) * batch.GROUP
    total = sum(tt)
    v = n_pairs / total
    line = {
        "impl": "reference", "metric": "registrations/sec", "value": v, "unit": "registrations/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 NN / f64 accumulate", "data": "synthetic",
        "config": {"workload": "BASELINE configs[3]: loop-closure candidate batch (GICP, 64k-pt VLP-16 pairs, 8 candidates per new keyframe), sharded by keyframe group",
                   "points_per_scan": 65536, "pairs_per_step": gps * batch.GROUP, "fitness_max_range": args.fitness_max_range},
        "cpu_baseline": {"value": v, "unit": "registrations/s", "cores": cores, "host_threads_available": host_threads(), "thread_sweep_pairs_per_s": table,
                         "kind": "port",
                         "sample": f"{n_pairs} candidate pairs ({gps} group(s) of 8 per step, {steps} steps) of the same workload: per group one kept target (kd-tree + "
                                   f"covariances), per candidate source kd-tree + covariances + align + getFitnessScore, as LoopDetector::matching does; oracle = "
                                   f"from-scratch OpenMP restatement of fast_gicp (upstream binaries cannot be built here)"},
        "e2e": {"value": v, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_reference(args, wl, rank):
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    timed = min(args.steps, 400)  # bounded sample: the CPU arm replays at most 400 frames so that any --steps ends within minutes
    frames = make_frames(wl["sensor"], 0, timed + args.warmup + 1)
    cores, sweep = best_thread_count(orc, frames, wl["method"], wl["params"])
    oracle_odometry(orc, frames[: args.warmup + 1], wl["method"], wl["params"], cores)  # first keyframe + warm-up
    # timed: continue the chain from a fresh keyframe at frame `warmup`
    times = oracle_odometry(orc, frames[args.warmup:], wl["method"], wl["params"], cores)[1:]
    total = sum(times)
    v = len(times) / total
    line = {
        "impl": "reference", "metric": "registrations/sec", "value": v, "unit": "registrations/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total / len(times) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 NN / f64 accumulate", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[{wl['config_index']}]: {args.workload}", "points_per_scan": int(frames[0].shape[0])},
        "cpu_baseline": {"value": v, "unit": "registrations/s", "cores": cores, "host_threads_available": host_threads(), "thread_sweep_frames_per_s": sweep,
                         "kind": "port",
                         "value_1thread": single_thread_figure(orc, frames[args.warmup:], wl["method"], wl["params"]),
                         "sample": f"{len(times)} consecutive frames of the same sequence (of --steps {args.steps}); oracle = from-scratch restatement of fast_gicp/ndt_omp (upstream binaries cannot be built here)"},
        "e2e": {"value": v, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def algorithmic_bytes(cls, n, m, stride_bytes):
    """SURVEY.md §8(d): compulsory bytes per launch of each kernel class (N source points, M target points)."""
    return {
        "knn_covariance": n * 16 + n * 48,
        "gicp_correspondences": 16 * (n + m) + 16 * n,          # src+tgt float4 once, seed read + corr/cpos/d2 writes
        "gicp_linearize": n * (16 + 4 + 48 + 48 + 16 + 48) + n * (4 + 48 + 16) + 29 * 8,  # point, cpos, C_A, C_B, target, M out; fused trial cost: cpos', M', target'
        "gicp_error": n * (16 + 4 + 48) + m * 16 + 8,
        "bvh_build": n * (stride_bytes + 16 + 4 + 16),
        "nn_fitness": n * 16 + m * 16 + 24,
        "ndt_derivatives": n * 16 + 43 * 8,  # + V*112 voxel records, added by the caller when V is known
        "ndt_voxel_build": m * 16,
    }.get(cls)


def whole_step_algorithmic_gbs(calls, n, m, stride_bytes, total_ms, steps):
    """All kernel classes of the timed region together: sum over classes of (calls x algorithmic bytes per launch) / timed wall time.
    Returns (GB/s, bytes per step, classes without a byte model) — the single-kernel roofline entry stays the headline figure."""
    total, unknown = 0, []
    for cls, c in calls.items():
        if not c:
            continue
        ab = algorithmic_bytes(cls, n, m, stride_bytes)
        if ab is None:
            unknown.append(cls)
            continue
        total += int(c) * int(ab)
    if total_ms <= 0 or steps <= 0:
        return None
    return total / (total_ms * 1e-3) / 1e9, total / steps, unknown


def dump_outputs(out_dir, outputs):
    """One out_dir/<name>.npy per value a caller of the timed path received: float32 arrays as returned, everything else as float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, v in outputs.items():
        a = np.asarray(v)
        np.save(os.path.join(out_dir, f"{name}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def run_b200(args, wl, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import hdl_graph_slam_b200 as pkg

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup
    nframes = K + W + 1
    frames = make_frames(wl["sensor"], rank * 37, nframes)  # each rank: its own stretch of the closed circuit (replica), own noise seeds
    n, stride_f = frames[0].shape
    stride_bytes = stride_f * 4
    host = torch.empty((nframes, n, stride_f), dtype=torch.float32, pin_memory=True)
    for i, f in enumerate(frames):
        host[i].copy_(torch.from_numpy(f))
    devbuf = host.to(dev)  # HBM-resident copy for the `value` arm
    torch.cuda.synchronize()

    params = {"registration_method": wl["method"]}
    params.update({k: v for k, v in wl["params"].items() if k.startswith("reg_")})
    results = {}
    # value: frames resident in HBM, no event recording; e2e: pinned host frames through the same call; profile: the value pass
    # again with per-kernel CUDA events on (recording two events per launch costs ~6 % of throughput, so the headline pass runs
    # without them) -> per-class kernel times and the roofline entry
    arms = ["value", "e2e"]
    if not args.no_prefetch and not args.no_anchor:
        arms.append("strict")  # the same K frames without announcing the next one: the strict call-by-call chain
    if not args.no_profile:
        arms.append("profile")
    for arm in arms:
        reg = pkg.select_registration_method(params, device_id=local_rank)
        if wl["method"] == "NDT_OMP":
            reg.close()
            cfg = pkg.default_config(pkg.B2R_METHOD_NDT)
            cfg.device_id = local_rank
            cfg.ndt_resolution = wl["params"].get("reg_resolution", 1.0)
            cfg.ndt_fixed_iterations = 30
            reg = pkg.Registration(cfg)
        odo = pkg.ScanMatchingOdometry(reg, keyframe_delta_trans=1.0, keyframe_delta_angle=1.0, keyframe_delta_time=10000.0)
        stream = torch.cuda.ExternalStream(reg.getStream(), device=dev)
        device_arm = arm not in ("e2e", "strict")  # strict chain: host buffers through the reference-facing call, like e2e
        base = devbuf.data_ptr() if device_arm else host.data_ptr()
        fbytes = n * stride_bytes

        prefetch = (not args.no_prefetch) and arm != "strict"

        def step(i):
            if prefetch and i + 1 < nframes:  # replay: the next scan is already in memory -> announce it (software pipelining)
                odo.prefetch_raw(base + (i + 1) * fbytes, n, stride_bytes, device=device_arm)
            return odo.matching_raw(0.1 * i, base + i * fbytes, n, stride_bytes, device=device_arm)

        for i in range(W + 1):  # first keyframe + W untimed warm-up frames
            step(i)
        reg.synchronize()
        reg.getStats(reset=True)
        reg.setProfiling(arm == "profile")
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank)
        if rank == 0 and arm == "value":
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        iters, conv, kf = 0, 0, 0
        t0 = time.perf_counter()
        for i in range(W + 1, W + 1 + K):
            st = step(i)
            iters += st["iterations"]; conv += int(st["converged"]); kf += int(st["keyframe_updated"])
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        per_rank = [ms]
        if world > 1:
            dist.barrier()
            allms = torch.zeros(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(allms, t)
            per_rank = [float(x) for x in allms.cpu()]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stats = reg.getStats()
        reg.setProfiling(False)
        clocks = None
        if rank == 0 and arm == "value":  # keep the same chain running (untimed) until nvidia-smi has sampled the load, then read the clocks
            sampler.hold(lambda k: step(W + 1 + (k % K)), reg.synchronize)
            clocks = sampler.stop()
        results[arm] = dict(ms=float(t.item()), per_rank_ms=per_rank, wall_ms=wall * 1e3, stats=stats, iters=iters, conv=conv, kf=kf, clocks=clocks,
                            last=st)
        odo.close()
        reg.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    rv, re_ = results["value"], results["e2e"]
    if args.dump_outputs:  # matching_error / inlier_fraction are left out: NaN, as the chain runs without publish_status
        dump_outputs(args.dump_outputs, {k: v for k, v in rv["last"].items() if k not in ("matching_error", "inlier_fraction")})
    value = world * K / (rv["ms"] * 1e-3)
    e2e = world * K / (re_["ms"] * 1e-3)
    launches = int(sum(rv["stats"]["launches"].values()))
    st = results["profile"]["stats"] if "profile" in results else rv["stats"]
    prof_ms = results["profile"]["ms"] if "profile" in results else rv["ms"]
    # dominant kernel class by CUDA-event time inside the timed region
    hbm, how = peaks()
    top = max(st["ms"], key=lambda k: st["ms"][k]) if any(st["ms"].values()) else None
    roofline = None
    if top and st["calls"][top]:
        per_launch_ms = st["ms"][top] / st["calls"][top]
        ab = algorithmic_bytes(top, n, n, stride_bytes)
        if ab:
            achieved = ab / (per_launch_ms * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": ncu_traffic(top),
                        "peak_source": f"of {how} (MEASURED_PEAKS.json hbm_gbs)" if how == "measured" else "of fallback (6.65 TB/s)",
                        "algorithmic_bytes_per_launch": ab, "avg_launch_us": per_launch_ms * 1e3, "launches_timed": st["calls"][top],
                        "share_of_step": st["ms"][top] / prof_ms,
                        "note": "single-pair working set (~9 MB) is L2-resident: this is the odometry chain's latency-bound figure; see DESIGN.md"}
    try:  # informational: the whole step's algorithmic bytes over the headline pass's time (never allowed to break the line)
        ws = whole_step_algorithmic_gbs(rv["stats"]["calls"], n, n, stride_bytes, rv["ms"], K)
        if roofline is not None and ws is not None:
            roofline["whole_step"] = {"achieved": ws[0], "unit": "GB/s", "frac": ws[0] / hbm, "algorithmic_bytes_per_step": ws[1],
                                      "classes_without_byte_model": ws[2],
                                      "note": "sum over kernel classes of launches x algorithmic bytes, divided by the timed region of the headline pass"}
    except Exception:  # noqa: BLE001
        pass
    kernel_ms = {k: round(v, 4) for k, v in st["ms"].items() if v > 0}
    # CPU baseline on a bounded sample of the same workload (rank 0, N = 1 only)
    cpu = None
    if world == 1 and args.cpu_sample > 0:
        from oracle import oracle as orc
        orc.build()
        sample = frames[W: W + 1 + max(args.cpu_sample, 6)]
        cores, sweep = best_thread_count(orc, sample, wl["method"], wl["params"])
        tt = oracle_odometry(orc, sample, wl["method"], wl["params"], cores)[1:]
        cpu = {"value": len(tt) / sum(tt), "unit": "registrations/s", "cores": cores, "host_threads_available": host_threads(), "thread_sweep_frames_per_s": sweep,
               "kind": "port",
               "value_1thread": single_thread_figure(orc, sample, wl["method"], wl["params"]),
               "sample": f"{len(tt)} consecutive frames of the timed sequence on the host cores (OpenMP oracle restating fast_gicp/ndt_omp; the upstream "
                         f"binaries cannot be built here)"}
    line = {
        "metric": "registrations/sec", "value": value, "unit": "registrations/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": rv["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 NN / f64 accumulate", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[{wl['config_index']}]: {args.workload}", "points_per_scan": int(n), "method": wl["method"],
                   "parallelism": f"replicas x{world} (odometry chain is sequential)",
                   "l2": "inputs larger than L2: every step consumes a distinct 2 MiB scan (K scans streamed once each); derived data is rebuilt per step",
                   "pipelining": "next scan announced to the engine (b2r_odometry_prefetch): its upload/BVH/covariances overlap the current align on a second stream" if not args.no_prefetch else "none (strict call-by-call chain)",
                   "mean_iterations": rv["iters"] / K, "converged_frac": rv["conv"] / K, "keyframe_switches": rv["kf"],
                   "strict_chain_value": (world * K / (results["strict"]["ms"] * 1e-3)) if "strict" in results else None,
                   "strict_chain_note": "same K frames from pinned host buffers WITHOUT b2r_odometry_prefetch: what a live scan_matching_odometry_nodelet "
                                        "(and the shipped pcl::Registration adapter) can issue; registrations/s"},
        "e2e": {"value": e2e, "unit": "registrations/s", "h2d_bytes_per_step": re_["stats"]["h2d_bytes"] / K, "d2h_bytes_per_step": re_["stats"]["d2h_bytes"] / K,
                "ms_per_step": re_["ms"] / K},
        "gpu_launches": launches,
        "clocks": rv["clocks"],
        "roofline": roofline,
        "cpu_baseline": cpu,
        "kernel_ms_in_timed_region": kernel_ms,
        "kernel_timing": {"pass": "same K steps repeated with per-launch CUDA events on the engine's streams", "ms_per_step": prof_ms / K},
        "wall_ms_per_step": rv["wall_ms"] / K,
        "per_rank_ms_per_step": [round(x / K, 4) for x in rv["per_rank_ms"]],
        "host_threads_visible": host_threads(),
    }
    if world == 1 and not args.no_anchor and wl["method"] == "FAST_GICP":
        # the 1-GPU anchor of the sharded workload (BASELINE configs[3]) that bench.py --gpus N measures for N > 1
        try:
            import types
            from hdl_graph_slam_b200 import batch
            a = types.SimpleNamespace(steps=3, warmup=3, pairs=args.pairs, fitness_max_range=args.fitness_max_range, no_profile=False)
            lb = batch.run_loop_batch(a, 0, 1, local_rank)
            line["loop_batch_n1"] = {k: lb[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "config", "e2e", "roofline", "gpu_launches",
                                                         "kernel_ms_in_timed_region")}
        except Exception as e:  # noqa: BLE001
            line["loop_batch_n1"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload is None:
        # the odometry chain cannot shard (frame k's guess is frame k-1's pose): at N > 1 measure the path that does
        args.workload = "loop_batch" if max(world, args.gpus) > 1 else "gicp_odometry_vlp16_64k"
    if args.dump_outputs and (args.impl != "b200" or args.workload not in WORKLOADS):
        sys.exit(f"--dump-outputs is implemented for the B200 arm of the odometry workloads ({', '.join(WORKLOADS)})")
    if args.steps is None:
        args.steps = 5 if (args.workload, args.impl) == ("loop_batch", "b200") else 200  # loop_batch: 5 timed passes of the whole batch
    if args.workload == "loop_batch":
        if args.impl == "reference":
            return run_reference_loop(args, rank)
        from hdl_graph_slam_b200 import batch
        args.warmup = max(args.warmup, 3) if args.warmup != 5 else 3
        return batch.bench_loop_batch(args, rank, world, local_rank)
    if args.workload in ("voxelgrid", "kitti_pipeline"):
        import bench_workloads
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"--workload {args.workload}: the CPU figure is this workload's own cpu_baseline object"}), flush=True)
            return
        fn = bench_workloads.bench_voxelgrid if args.workload == "voxelgrid" else bench_workloads.bench_kitti_pipeline
        return fn(args, rank, world, local_rank)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl, rank)
    run_b200(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
