#!/usr/bin/env python
"""bench.py -- scans/sec of the per-scan hot path (SurfelMapping::processScan, loop closure off) on synthetic
HDL-64E-shaped scans: 64 x 2048 range images, exactly 10 Gauss-Newton iterations (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            # N > 1: launched under torchrun, one rank per GPU
  python bench.py --impl reference --steps K --warmup W    # the CPU restatement of the reference (oracle/, OpenMP) on the host
                                                           # cores; --reference-kind itself: the reference's own classes
                                                           # and shaders on the single-thread software GL (oracle/_ref)

One step = one scan through the whole path (K1-K3 preprocessing, model rendering, 10 x (K5 + GN step), post-ICP
rendering + statistics pass, K6 map update, model re-render). `value` is measured with the scans already resident in
HBM; `e2e` goes through the C ABI with pinned HOST buffers (H2D of the scan and D2H of the pose / sums inside the
timed region). Every pass first pre-rolls the map with --preroll scans (steady-state map size, SURVEY.md 8d) and the
--warmup scans, untimed. N > 1 runs one independent sequence per GPU (weak scaling, no data-path collective) and adds a
`striped` record: BASELINE.json configs[3] (128x4096, 15 iterations, row-striped K5 with the in-kernel peer-memory
all-reduce) on the same GPUs, against the same sequence without striping. Prints ONE JSON line on rank 0.
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from semantic_suma_b200 import synth  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: KITTI-shaped 64x2048, geometric SuMa (no labels), exactly 10 ICP iterations
    "hdl64_2048_geometric": dict(width=2048, height=64, fov_up=3.0, fov_down=-25.0, semantic=False, iters=10),
    # configs[2]: semantic-weighted ICP + label-consistent fusion
    "hdl64_2048_semantic": dict(width=2048, height=64, fov_up=3.0, fov_down=-25.0, semantic=True, iters=10),
    # configs[0]: the plumbing case
    "hdl64_900_geometric": dict(width=900, height=64, fov_up=3.0, fov_down=-25.0, semantic=False, iters=10),
    # configs[3]: Ouster-128-style
    "ouster128_4096_geometric": dict(width=4096, height=128, fov_up=22.5, fov_down=-22.5, semantic=False, iters=15),
}


def param_kwargs(w):
    return dict(data_width=w["width"], data_height=w["height"], model_width=w["width"], model_height=w["height"],
                data_fov_up=w["fov_up"], data_fov_down=w["fov_down"], model_fov_up=w["fov_up"],
                model_fov_down=w["fov_down"], max_iterations=w["iters"], stopping_threshold=0.0, delta=0.0)


def _gen_one(job):
    w, seed, frame, pose = job
    sc = synth.Scene(width=w["width"], height=w["height"], fov_up=w["fov_up"], fov_down=w["fov_down"],
                     semantic=w["semantic"], seed=seed)
    return sc.scan(frame, pose)


def generate_scans(w, n_frames, seed):
    poses = synth.trajectory(n_frames)
    jobs = [(w, seed, f, poses[f]) for f in range(n_frames)]
    workers = max(1, min(32, (os.cpu_count() or 2) // max(1, int(os.environ.get("WORLD_SIZE", "1"))) - 1))
    if workers > 1 and n_frames > 4:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(workers) as pool:
            return pool.map(_gen_one, jobs, chunksize=2)
    return [_gen_one(j) for j in jobs]


class ClockSampler(threading.Thread):
    """samples SM clock / power / throttle reasons during the timed region (B200_PROFILING.md, clocks line).
    Uses NVML in-process (nvidia_ml_py): spawning nvidia-smi every 100 ms perturbs a 50 ms timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        except Exception:  # noqa: BLE001
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:  # noqa: BLE001
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        flags = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        return [sm, mx, pw] + [bool(r & v) for v in (flags["hw_slowdown"], flags["hw_thermal_slowdown"],
                                                     flags["sw_thermal_slowdown"], flags["sw_power_cap"])]

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        return [float(f[0]), float(f[1]), float(f[2])] + [x.lower().startswith("active") for x in f[3:7]]

    def run(self):  # thread mode (not used by the timed passes any more, see sample_once)
        while not self.stop_flag:
            self.sample_once()
            time.sleep(0.05 if self.nvml else 0.2)

    def sample_once(self):
        """One sample, taken synchronously by the caller BETWEEN two timed steps in the middle of the timed region (a
        concurrent NVML thread polling every few ms during a 10 ms pass was the prime suspect for the isolated multi-ms
        steps that the 4- and 8-GPU runs showed on single ranks -- eight processes queueing on the driver's global lock)."""
        try:
            self.samples.append(self._sample_nvml() if self.nvml else self._sample_smi())
        except Exception:  # noqa: BLE001
            pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i] for s in self.samples)]
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": max(s[1] for s in self.samples),
                "power_w_max": round(max(s[2] for s in self.samples), 1), "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self.nvml else "nvidia-smi"}


ITERS = [10]  # Gauss-Newton iterations of the workload (set by run_native)


def algorithmic_bytes(kernel, P, S, N, semantic):
    """compulsory HBM bytes of one launch (DESIGN.md 'Kernels and their rooflines'; SURVEY.md 8d)"""
    t = {
        "fill_u64": 8 * P, "project_scatter": 16 * N, "preprocess_tile": 8 * P + 16 * N + (48 + 16) * P,
        # the persistent Gauss-Newton launch re-reads the six range images every iteration (SURVEY.md 8d: 64P / 96P per
        # iteration); icp_post = the statistics pass of updatePose (one iteration's worth)
        "icp_fused": ITERS[0] * (96 if semantic else 64) * P, "icp_post": (96 if semantic else 64) * P,
        "icp_jacobian": (96 if semantic else 64) * P,
        "render_scatter": 48 * S, "render_resolve": 3 * 8 * P + 4 * 48 * P,
        "index_scatter": 48 * S, "radius": 48 * P, "update_surfels": 129 * S, "gen_surfels": 84 * P,
        "compact_scatter": 129 * S, "scan_blocks": 8 * (S // 256 + 1), "pose_products": 128 * 100,
    }
    return float(t.get(kernel, 0))


def pin_to_gpu_numa_node(local_rank):
    """run this rank on the CPUs next to its GPU (nvidia-smi topo 'CPU Affinity'): launches and pinned copies of GPUs
    4-7 otherwise cross the socket interconnect. Returns the cpu list used (or None)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d-%d (%d cpus)" % (min(cpus), max(cpus), len(cpus))
    except Exception:  # noqa: BLE001
        pass
    return None


def run_native(args, w, rank, world, local_rank):
    import torch
    from semantic_suma_b200 import api

    ITERS[0] = w["iters"]
    pre = args.preroll + args.warmup            # scans processed before the timed region of every pass
    n_frames = pre + args.steps
    scans = generate_scans(w, n_frames, seed=1337 + 1000 * rank)
    striped_scans = None
    if world > 1 and not args.no_striped:  # generated now: the worker pool forks, which must happen before CUDA is up
        striped_scans = generate_scans(WORKLOADS["ouster128_4096_geometric"], STRIPED_PRE + STRIPED_STEPS, seed=4242)
    numa = pin_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # communicator set-up (lazy: first collective) long before anything is timed
        warm = torch.zeros(1, device="cuda")
        dist.all_reduce(warm)
        dist.barrier()
        torch.cuda.synchronize()
    pp = api.default_params(**param_kwargs(w))
    slam = api.SurfelMapping(pp, device=local_rank)
    ctx = slam.ctx
    stream = torch.cuda.ExternalStream(ctx.stream(), device=local_rank)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    sem = w["semantic"]

    dev = [(torch.from_numpy(p).cuda(), torch.from_numpy(l).cuda() if sem else None,
            torch.from_numpy(q).cuda() if sem else None) for p, l, q in scans]
    pin = [(torch.from_numpy(p).pin_memory(), torch.from_numpy(l).pin_memory() if sem else None,
            torch.from_numpy(q).pin_memory() if sem else None) for p, l, q in scans]
    h2d = sum(int(p.numel() * 4 + (l.numel() * 4 + q.numel() * 4 if sem else 0)) for p, l, q in pin[pre:])
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def feed(bufs, f, on_device, prefetch_next=True):
        if args.prefetch and not on_device and prefetch_next and f + 1 < len(bufs):
            # host buffers: stage the NEXT scan on the copy stream while this one is processed (sb_prefetch_scan)
            pn, ln, qn = bufs[f + 1]
            slam.prefetch_scan_raw(pn.data_ptr(), ln.data_ptr() if sem else 0, qn.data_ptr() if sem else 0, pn.shape[0])
        p, l, q = bufs[f]
        slam.process_scan_raw(p.data_ptr(), l.data_ptr() if sem else 0, q.data_ptr() if sem else 0, p.shape[0], on_device)

    def preroll(bufs, on_device):
        """map pre-rolled to the steady state of SURVEY.md 8d (independent of --steps / --warmup) + the warm-up scans"""
        slam.reset()
        for f in range(pre):  # the first timed scan is NOT staged ahead: its host-to-device copy belongs to the timed region
            feed(bufs, f, on_device, prefetch_next=f + 1 < pre)
        ctx.synchronize()

    def one_pass(bufs, on_device, sampler=None):
        preroll(bufs, on_device)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        launches0 = ctx.launch_count()
        barrier()
        host_split = []
        gc_was = gc.isenabled()
        gc.disable()  # no collector pause inside a 10 ms pass
        t_wall = time.time()
        for i in range(args.steps):
            with torch.cuda.stream(stream):
                flush.zero_()  # L2 flush between timed steps (not timed)
            ev[i][0].record(stream)
            feed(bufs, pre + i, on_device)
            if not on_device:
                slam.getCurrentPose()  # the step's result, read on the host
            ev[i][1].record(stream)
            st = slam.getStatistics()
            host_split.append((st["preprocessing-time"], st["icp-time"], st["mapping-time"]))
            if sampler and i == args.steps // 2:
                sampler.sample_once()  # clocks / throttle reasons in the middle of the timed region, between two steps
        barrier()
        t_wall = time.time() - t_wall
        if gc_was:
            gc.enable()
        ms = [a.elapsed_time(b) for a, b in ev]
        worst = max(range(len(ms)), key=lambda j: ms[j])
        one_pass.worst_step = {"step": worst, "device_ms": round(ms[worst], 4),
                               "host_enqueue_ms": round(1e3 * host_split[worst][0], 4),
                               "host_wait_ms": round(1e3 * host_split[worst][1], 4),
                               "host_post_ms": round(1e3 * host_split[worst][2], 4)}
        total_ms = worst_ms = float(sum(ms))
        if dist is not None:
            t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            worst_ms = float(t.item())
        return worst_ms, ctx.launch_count() - launches0, t_wall, ms

    # every GPU busy for >= 0.6 s right before the first timed pass: clocks of GPUs that idled are up, the caches of the
    # host launch path are warm (SCALE_r01: the first pass caught a transient on the slowest rank)
    t0 = time.time()
    while True:
        preroll(dev, True)
        if time.time() - t0 > 0.6:
            break
    sampler = ClockSampler(local_rank)
    ms_dev, launches, wall_dev, per_step = one_pass(dev, True, sampler)
    worst_dev = dict(one_pass.worst_step)
    ms_e2e, _, wall_e2e, per_step_e2e = one_pass(pin, False)
    if args.dump_outputs and rank == 0:
        dump_outputs(slam, args.dump_outputs)
    surfels = slam.getMap().size()
    gt = np.linalg.inv(synth.trajectory(1)[0]) @ synth.trajectory(n_frames)[-1]
    drift = float(np.linalg.norm(slam.getCurrentPose()[:3, 3] - gt[:3, 3]))
    mine = {"rank": rank, "step_ms_min_med_max": [round(min(per_step), 4), round(statistics.median(per_step), 4),
                                                  round(max(per_step), 4)],
            "e2e_step_ms_med": round(statistics.median(per_step_e2e), 4), "slowest_step": worst_dev,
            "clocks": sampler.summary(), "numa_cpus": numa}
    per_rank = [mine]
    if dist is not None:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    # per-kernel device time with CUDA events on the launching stream, over the same timed frames
    roofline = None
    kernel_table = {}
    if rank == 0 and not args.no_profile:
        try:  # the per-kernel table explains the headline; a failure in it must not cost the line
            preroll(dev, True)
            ctx.profile(True)
            s_sum = 0
            per_step_prof = []
            for i in range(args.steps):
                with torch.cuda.stream(stream):
                    flush.zero_()
                s_sum += slam.getMap().size()
                feed(dev, pre + i, True)
                per_step_prof.append(ctx.profile_collect())
            ctx.profile(False)
            # per kernel class: median over the steps of the step's mean launch time (one disturbed launch -- another
            # process initialising on the box, a clock sample -- must not move a 15 us kernel's figure), times its launches
            prof = {}
            for k in {k for st in per_step_prof for k in st}:
                per = [st[k][0] / st[k][1] for st in per_step_prof if k in st and st[k][1] > 0]
                cnt = sum(st[k][1] for st in per_step_prof if k in st)
                if per and cnt:
                    prof[k] = (statistics.median(per) * cnt, cnt)
            tot = sum(v[0] for v in prof.values())
            P = w["width"] * w["height"]
            S_avg = s_sum / max(1, args.steps)
            N_avg = float(np.mean([p.shape[0] for p, _, _ in scans[pre:]]))
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:  # noqa: BLE001
                pass
            peak = float(peaks.get("hbm_gbs", 6650.0))
            for k, (ms, cnt) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
                b = algorithmic_bytes(k, P, S_avg, N_avg, sem)
                us = 1e3 * ms / cnt
                kernel_table[k] = {"launches_per_step": round(cnt / args.steps, 2), "avg_us": round(us, 2),
                                   "share": round(ms / tot, 4), "gbps": round(b / (us * 1e-6) / 1e9, 1) if us > 0 else None}
            top = max(prof.items(), key=lambda kv: kv[1][0])[0]
            us = 1e3 * prof[top][0] / prof[top][1]
            ach = algorithmic_bytes(top, P, S_avg, N_avg, sem) / (us * 1e-6) / 1e9
            traffic, traffic_src, traffic_S = None, None, None
            try:  # DRAM bytes of this kernel from the committed ncu --set full capture (profiles/ncu_traffic.py)
                tj = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
                traffic = tj["kernels"][top]["dram_bytes_per_launch"]
                traffic_src = tj.get("source")
                traffic_S = tj.get("surfels_at_capture")
            except Exception:  # noqa: BLE001
                pass
            roofline = {"kernel": top, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                        "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                        "traffic_at_surfels": traffic_S,  # the ncu capture's map size (S of this run: surfels_avg below)
                        "algorithmic_bytes_per_launch": int(algorithmic_bytes(top, P, S_avg, N_avg, sem)),
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                        "avg_launch_us": round(us, 2), "surfels_avg": int(S_avg),
                        "step_share": kernel_table[top]["share"]}
        except Exception as e:  # noqa: BLE001
            roofline = {"error": "per-kernel pass failed: %s: %s" % (type(e).__name__, str(e)[:200])}
    if dist is not None:
        dist.barrier()  # the other ranks stay quiet while rank 0 takes the per-kernel times
    slam.ctx.close()
    del dev, pin
    torch.cuda.empty_cache()

    out = None
    if rank == 0:
        # the CPU baseline is timed at N = 1 only (rank 0); the N > 1 lines carry null
        cpu = None
        if not (args.no_cpu_baseline or world > 1):
            try:
                cpu = cpu_baseline(w, scans, budget_s=args.cpu_budget)
            except Exception as e:  # noqa: BLE001 -- the GPU figures above are complete; report why the CPU arm is missing
                cpu = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
        value = world * args.steps / (ms_dev * 1e-3)
        e2e_value = world * args.steps / (ms_e2e * 1e-3)
        out = {
            "metric": "scans_per_sec", "value": round(value, 2), "unit": "scans/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_dev / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "range_image": "%dx%d" % (w["height"], w["width"]),
                       "icp_iterations": w["iters"], "semantic": sem, "sequences": world,
                       "parallelism": "one sequence per GPU, no data-path collective",
                       "map_preroll_scans": args.preroll, "surfels_end": int(surfels), "pose_drift_m": round(drift, 4),
                       "l2": "flushed between timed steps (256 MiB memset, untimed)",
                       "gpu_preroll": ">= 0.6 s of scans on every rank before the timed pass",
                       "per_rank": per_rank,
                       "timing": "CUDA events on the library's stream around every step, summed; max over ranks",
                       "reference_defaults": "config/default.xml except image size, max iterations, eps=delta=0"},
            "e2e": {"value": round(e2e_value, 2), "unit": "scans/s", "ms_per_step": round(ms_e2e / args.steps, 4),
                    "h2d_bytes_per_step": int(h2d / args.steps) + 128, "d2h_bytes_per_step": 8192 + 64,
                    "wall_s": round(wall_e2e, 3), "input_prefetch": bool(args.prefetch)},
            "gpu_launches": int(launches),
            "clocks": per_rank[0]["clocks"],
            "roofline": roofline, "kernels": kernel_table, "cpu_baseline": cpu,
        }
    if dist is not None and not args.no_striped:
        # The extra record must never cost the replica line: it runs AFTER that line is complete, under a per-rank
        # deadline. If a rank fails or the ranks lose each other (one raised, the others wait in a collective), every
        # rank's deadline fires: rank 0 prints the line it already has (striped = the error) and all ranks exit 0.
        guard = StripedGuard(rank, out, args.striped_deadline)
        guard.start()
        try:
            striped = striped_record(striped_scans, rank, world, local_rank, dist)
        except Exception as e:  # noqa: BLE001
            striped = {"error": "%s: %s" % (type(e).__name__, str(e)[:300]), "rank": rank}
        errs = [None] * world
        dist.all_gather_object(errs, striped.get("error") if isinstance(striped, dict) else "no record")
        if rank == 0:
            bad = [(r, e) for r, e in enumerate(errs) if e]
            out["striped"] = striped if not bad else {"error": "; ".join("rank %d: %s" % be for be in bad)}
        dist.barrier()
        guard.cancel()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return out


DUMP_SURFELS = 1 << 17  # at most this many surfel records (a fixed, seeded sample of the map) go to surfels.npy


def dump_outputs(slam, out_dir):
    """what a caller of processScan receives after the last timed step, as DIR/<name>.npy (float32 / float64, < 64 MB):
    the pose, the ICP statistics, the surfel map (count + sampled records) and the current data / model frames"""
    os.makedirs(out_dir, exist_ok=True)
    st = slam.getStatistics()
    surf = slam.getMap().getAllSurfels()
    n = surf.shape[0]
    idx = np.arange(n) if n <= DUMP_SURFELS else np.sort(np.random.default_rng(0).choice(n, DUMP_SURFELS, replace=False))
    out = {"pose": slam.getCurrentPose(),
           "icp_statistics": np.array([st[k] for k in ("num_iterations", "F", "inlier", "outlier", "invalid",
                                                       "inlier_residual", "track_loss")], np.float64),
           "surfel_count": np.array([n], np.float64),
           "surfel_sample_index": idx.astype(np.float64),
           "surfels": np.stack([surf[f][idx].astype(np.float32) for f in surf.dtype.names], 1)}
    for name, frame in (("current_frame", slam.getCurrentFrame()), ("current_model_frame", slam.getCurrentModelFrame())):
        for part, a in zip(("vertex", "normal", "semantic"), frame.maps()):
            out["%s_%s" % (name, part)] = a
    for k, v in list(out.items()):
        # Every file holds finite numbers only. A non-finite element is written as 0, and <name>_nonfinite.npy lists it
        # as (flat index, 1 = NaN / 2 = +inf / 3 = -inf). Such elements are part of the result: the reference's
        # slerp (update_surfels.vert:113-124) divides by sin(0) when a surfel's normal equals the measured one, which
        # leaves that surfel's normal NaN.
        bad = np.flatnonzero(~np.isfinite(v))
        if bad.size:
            flat = v.reshape(-1)
            code = np.where(np.isnan(flat[bad]), 1, np.where(flat[bad] > 0, 2, 3))
            out[k + "_nonfinite"] = np.stack([bad, code], 1).astype(np.float64)
            out[k] = np.where(np.isfinite(v), v, 0).astype(v.dtype)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


class StripedGuard(threading.Thread):
    """deadline for the optional `striped` record of the N > 1 runs (see run_native)"""

    def __init__(self, rank, out, seconds):
        super().__init__(daemon=True)
        self.rank, self.out, self.seconds = rank, out, seconds
        self.done = threading.Event()

    def cancel(self):
        self.done.set()

    def run(self):
        if self.done.wait(self.seconds):
            return
        if self.rank == 0 and self.out is not None:
            self.out["striped"] = {"error": "no result within %.0f s (a rank failed or the ranks lost each other); the "
                                            "replica figures above were complete before it started" % self.seconds}
            sys.stdout.write(json.dumps(self.out) + "\n")
            sys.stdout.flush()
        os._exit(0)


STRIPED_PRE, STRIPED_STEPS = 10, 10


def striped_record(scans, rank, world, local_rank, dist):
    """BASELINE.json configs[3] on the same N GPUs: 128x4096 Ouster-style scans, 15 Gauss-Newton iterations, ONE sequence,
    the K5 reduction striped over image rows, the 32 sums exchanged inside the persistent kernel over peer memory
    (NVLink); the map is replicated. Measured against the same sequence run by every rank on its own (all rows, no
    exchange); poses must be bit-identical across ranks and between both runs."""
    import torch
    from semantic_suma_b200 import api, stripes
    w = WORKLOADS["ouster128_4096_geometric"]
    pre, steps = STRIPED_PRE, STRIPED_STEPS
    pp = api.default_params(**param_kwargs(w))
    dev = [torch.from_numpy(p).cuda() for p, _, _ in scans]
    torch.cuda.synchronize()
    res = {}
    poses = {}
    for mode in ("solo", "striped"):
        slam = api.SurfelMapping(pp, device=local_rank)
        ctx = slam.ctx
        rows = (0, w["height"])
        if mode == "striped":
            rows = stripes.setup_comm(ctx, dist, fused=True)
        stream = torch.cuda.ExternalStream(ctx.stream(), device=local_rank)
        for f in range(pre):
            slam.process_scan_raw(dev[f].data_ptr(), 0, 0, dev[f].shape[0], True)
        ctx.synchronize()
        torch.cuda.synchronize()
        dist.barrier()
        ctx.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            slam.process_scan_raw(dev[pre + i].data_ptr(), 0, 0, dev[pre + i].shape[0], True)
        e1.record(stream)
        ctx.synchronize()
        prof = ctx.profile_collect()
        ctx.profile(False)
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gn_ms, gn_n = prof.get("icp_fused", (0.0, 1))
        # the long launch is the 15-iteration minimisation; the short one the statistics pass
        res[mode] = {"ms_per_scan": round(float(t.item()) / steps, 4), "rows": list(rows),
                     "gn_launch_us_avg": round(1e3 * gn_ms / max(gn_n, 1), 2), "gn_launches_per_scan": round(gn_n / steps, 2)}
        poses[mode] = slam.getCurrentPose().tobytes()
        slam.ctx.close()
    allp = [None] * world
    dist.all_gather_object(allp, (poses["solo"], poses["striped"]))
    identical = all(a == allp[0][0] and b == allp[0][0] for a, b in allp)
    it = w["iters"]
    # per scan: one GN_MAIN launch (15 iterations) + one GN_POST launch (1 statistics pass): 16 passes
    d_us = (res["striped"]["gn_launch_us_avg"] - res["solo"]["gn_launch_us_avg"]) * 2.0 / (it + 1)
    return {"workload": "ouster128_4096_geometric", "icp_iterations": it, "n_gpus": world, "scans": steps,
            "exchange": "32 int64 sums per iteration, stored into every rank's mailbox and summed in-kernel (peer memory)",
            "solo": res["solo"], "striped": res["striped"],
            "speedup_vs_solo": round(res["solo"]["ms_per_scan"] / res["striped"]["ms_per_scan"], 4),
            "gn_pass_us_delta_striped_minus_solo": round(d_us, 3),
            "poses_bit_identical_across_ranks_and_modes": bool(identical)}


def physical_cores_per_socket():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("cpu cores"):
                return int(line.split(":")[1])
    except Exception:  # noqa: BLE001
        pass
    return os.cpu_count() or 1


def oracle_threads():
    """a FIXED rule, so that the CPU arm does not swing between boxes: the physical cores of one socket, at most 64 (the
    oracle's cap) and at most what this process may use"""
    return max(1, min(physical_cores_per_socket(), 64, len(os.sched_getaffinity(0))))


def cpu_baseline(w, scans, budget_s=15.0, max_frames=None):
    """the CPU restatement of the reference (oracle/) on a bounded sample of the same scans: OpenMP on the physical cores
    of one socket, plus the single-thread figure BASELINE.json's north_star names"""
    from oracle import oracle as O
    po = O.default_params(**param_kwargs(w))
    O.set_threads(1)
    sl = O.Slam(po)
    t0 = time.time()
    n1 = 0
    for p, l, q in scans[:4]:
        sl.process_scan(p, l, q)
        n1 += 1
        if time.time() - t0 > 0.35 * budget_s:
            break
    single = n1 / (time.time() - t0)
    threads = O.set_threads(oracle_threads())
    sl = O.Slam(po)
    t0 = time.time()
    n = 0
    for p, l, q in scans:
        sl.process_scan(p, l, q)
        n += 1
        if time.time() - t0 > budget_s or (max_frames and n >= max_frames):
            break
    dt = time.time() - t0
    return {"value": round(n / dt, 3), "unit": "scans/s", "cores": threads, "kind": "port",
            "sample": "first %d scans of the same synthetic sequence (map grows from empty), oracle/ C port, %d OpenMP "
                      "threads = physical cores of one socket" % (n, threads),
            "single_thread": {"value": round(single, 3), "unit": "scans/s", "cores": 1, "sample": "first %d scans" % n1},
            "seconds": round(dt, 2), "host_cpus": os.cpu_count()}


def reference_itself_sample(w, scans, budget_s=12.0, max_frames=6):
    """informational: the reference's OWN classes and shaders (oracle/_ref/libsuma_ref_full.so -- core/*.cpp compiled where
    they lie, running on a single-thread software GL) on the first scans of the sequence. Not the timed arm: a GL
    emulation says nothing about the reference's speed on a GPU; the multi-threaded port above is the stricter baseline."""
    try:
        from oracle import oracle as O
        from oracle import ref as R
        if not R.full_available():
            return None
        sys.stdout.flush()
        saved, null = os.dup(1), os.open(os.devnull, os.O_WRONLY)
        os.dup2(null, 1)  # the reference's classes print progress to stdout; this process prints ONE JSON line there
        try:
            f = R.Full(O.default_params(**param_kwargs(w)))
            t0 = time.time()
            n = 0
            for p, l, q in scans[:max_frames]:
                f.process_scan(p, l, q)
                n += 1
                if time.time() - t0 > budget_s:
                    break
            dt = time.time() - t0
            del f
        finally:
            os.dup2(saved, 1)
            os.close(saved)
            os.close(null)
        return {"value": round(n / dt, 3), "unit": "scans/s", "cores": 1, "kind": "reference",
                "sample": "first %d scans (map grows from empty): SurfelMapping::processScan of the reference itself, its "
                          "GLSL shaders transpiled, on a software GL" % n}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)[:200]}


def run_reference_itself(args, w, world, scans, pre):
    """--impl reference --reference-kind itself: SurfelMapping::processScan of the reference (oracle/_ref/libsuma_ref_full.so)
    on the same pre-rolled sequence; single thread, software GL"""
    from oracle import oracle as O
    from oracle import ref as R
    sys.stdout.flush()
    saved, null = os.dup(1), os.open(os.devnull, os.O_WRONLY)
    os.dup2(null, 1)  # the reference's classes print to stdout
    try:
        f = R.Full(O.default_params(**param_kwargs(w)))
        for i in range(pre):
            f.process_scan(*scans[i])
        t0 = time.time()
        done = 0
        for i in range(args.steps):
            f.process_scan(*scans[pre + i])
            done += 1
            if time.time() - t0 > args.ref_budget:
                break
        dt = time.time() - t0
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(null)
    v = done / dt
    return {
        "impl": "reference", "metric": "scans_per_sec", "value": round(v, 3), "unit": "scans/s", "n_gpus": world,
        "steps": done, "warmup": args.warmup, "ms_per_step": round(1e3 * dt / done, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "range_image": "%dx%d" % (w["height"], w["width"]),
                   "icp_iterations": w["iters"], "semantic": w["semantic"], "map_preroll_scans": args.preroll,
                   "note": "the reference's own core classes and GLSL shaders (compiled / transpiled from /root/reference, "
                           "oracle/_ref) on a single-thread software GL -- an emulation of its GPU path, not its speed on a GPU"},
        "cpu_baseline": {"value": round(v, 3), "unit": "scans/s", "cores": 1, "kind": "reference",
                         "sample": "%d scans after %d pre-roll + %d warm-up scans, one thread" % (done, args.preroll, args.warmup),
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": round(v, 3), "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def run_reference(args, w, rank, world):
    """--impl reference: the reference has no CPU (or buildable GL) path in this environment; the arm times the
    oracle's restatement of it (C + OpenMP, thread-count independent results) on the same workload, same pre-rolled map."""
    if rank != 0:
        return None
    pre = args.preroll + args.warmup
    scans = generate_scans(w, pre + args.steps, seed=1337)
    if args.reference_kind == "itself":
        return run_reference_itself(args, w, world, scans, pre)
    from oracle import oracle as O
    threads = O.set_threads(oracle_threads())
    po = O.default_params(**param_kwargs(w))
    sl = O.Slam(po)
    for f in range(pre):
        sl.process_scan(*scans[f])
    t0 = time.time()
    done = 0
    for i in range(args.steps):
        sl.process_scan(*scans[pre + i])
        done += 1
        if time.time() - t0 > args.ref_budget:
            break
    dt = time.time() - t0
    v = done / dt
    return {
        "impl": "reference", "metric": "scans_per_sec", "value": round(v, 3), "unit": "scans/s", "n_gpus": world,
        "steps": done, "warmup": args.warmup, "ms_per_step": round(1e3 * dt / done, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "range_image": "%dx%d" % (w["height"], w["width"]),
                   "icp_iterations": w["iters"], "semantic": w["semantic"], "map_preroll_scans": args.preroll,
                   "note": "no GL/EGL on the box: the reference's OpenGL path cannot run on the GPU. Timed here: the CPU "
                           "restatement in oracle/ (kind=port, OpenMP), which equals the reference's own classes + shaders "
                           "run on a software GL bit for bit (oracle/_ref, tests/test_ref_full.py); that run itself is "
                           "reported as cpu_baseline.reference_itself (single thread, far slower -- not the timed arm)"},
        "cpu_baseline": {"value": round(v, 3), "unit": "scans/s", "cores": threads, "kind": "port",
                         "sample": "%d scans after %d pre-roll + %d warm-up scans, %d OpenMP threads (physical cores of "
                                   "one socket)" % (done, args.preroll, args.warmup, threads),
                         "host_cpus": os.cpu_count(), "reference_itself": reference_itself_sample(w, scans)},
        "e2e": {"value": round(v, 3), "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    if os.environ.get("SUMA_B200_WATCHDOG"):  # debugging aid: dump the Python stacks if the run hangs
        import faulthandler
        faulthandler.enable()
        faulthandler.dump_traceback_later(float(os.environ["SUMA_B200_WATCHDOG"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="hdl64_2048_geometric", choices=sorted(WORKLOADS))
    ap.add_argument("--preroll", type=int, default=60,
                    help="scans processed (untimed) before the warm-up scans of every pass, in both arms: the map reaches the "
                         "steady-state size of SURVEY.md 8d (~1e6 surfels) independent of --steps / --warmup")
    ap.add_argument("--no-striped", action="store_true",
                    help="N > 1: skip the extra `striped` record (128x4096, 15 iterations, row-striped K5 with the in-kernel "
                         "peer-memory all-reduce, BASELINE.json configs[3])")
    ap.add_argument("--striped-deadline", type=float, default=240.0,
                    help="N > 1: seconds the `striped` record may take before the line is printed without it")
    ap.add_argument("--no-prefetch", dest="prefetch", action="store_false",
                    help="e2e pass: do not stage scan i+1 on the copy stream while scan i is processed (sb_prefetch_scan); "
                         "with or without it every copy is inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (pose, statistics, surfels, frames) as "
                         "DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--ref-budget", type=float, default=240.0)
    ap.add_argument("--reference-kind", default="port", choices=["port", "itself"],
                    help="--impl reference: 'port' times oracle/ (C + OpenMP, the stricter baseline, default); 'itself' times "
                         "the reference's own classes and shaders on the single-thread software GL (oracle/_ref)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        print("bench.py: --gpus %d needs torchrun (python -m torch.distributed.run --nproc-per-node %d ...)" %
              (args.gpus, args.gpus), file=sys.stderr)
        sys.exit(2)
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        out = run_reference(args, w, rank, world)
    else:
        out = run_native(args, w, rank, world, local_rank)
    if rank == 0 and out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
