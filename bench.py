#!/usr/bin/env python
"""bench.py -- ray-correspondences/s (and MICP-L iters/s) of the ray-casting-correspondence path on B200.

Workload (BASELINE.json configs[1], "C2"): MICP-L SphereCorrector, 1 pose x 128x1024 spherical scan on the 1 000 000-triangle
building mesh.  One step = one MICPLocalizationNode::correctOnce for that sensor: 1 find (131 072 rays traced) + 5 x (P2L cross
statistics -> Umeyama -> compose), rmcl_ros/src/nodes/micp_localization.cpp:899-984.
  value : device-resident step (dataset already in HBM), timed with CUDA events on the launching stream, L2 flushed between steps.
  e2e   : the same step through the C-ABI entry b2_rcc_correct_once_ranges with the scan in pinned HOST memory: H2D of the ranges and
          D2H of the result inside the timed region (host wall clock around the synchronous call).
N > 1 (torchrun): poses are sharded, one pose (one sensor) per GPU, map replicated, no data-path collective ("weak" scaling).

  python bench.py --gpus 1 --steps 200 --warmup 20
  python bench.py --gpus 1 --steps 200 --warmup 20 --dump-outputs /tmp/out    # + the last timed step's result as .npy files
  python bench.py --impl reference ...      # the reference's CPU path (oracle port: Embree/rmagine are not buildable here) on the host cores
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FACES = 1_000_000
ITERATIONS = 5
MAX_DIST, ADAPTIVE_MIN = 1.0, 0.15


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)      # ~0.1 s per timed region: long enough for several nvidia-smi samples inside it
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads (C3 particle filter, v1 batched correct)")
    ap.add_argument("--faces", type=int, default=N_FACES)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (the correctOnce result: "
                    "new pose, pose delta, merged statistics) to DIR/<name>.npy; same arguments, same inputs, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def dump_outputs(path, records):
    """One DIR/<record>_<field>.npy per field of each returned record: float32 fields as they are, integer fields (n_meas, stamp) as float64."""
    os.makedirs(path, exist_ok=True)
    for name, rec in records.items():
        for field in rec.dtype.names:
            v = np.asarray(rec[field])
            np.save(os.path.join(path, f"{name}_{field}.npy"), v if v.dtype == np.float32 else v.astype(np.float64))


def rank_pose(synth, rank):
    """pose guess of this rank's sensor: T_gt o (0.1,-0.05,0.2 m, yaw 3 deg) o a small rank-dependent shift"""
    T = synth.compose(synth.building_gt_pose(), synth.scenario_pose_offset())
    if rank:
        T = synth.compose(T, synth.make_transform((0.01 * rank, -0.007 * rank, 0.0), (0, 0, 0.002 * rank)))
    return T


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md 'clocks' line)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_indices):
        self.gpus = ",".join(str(g) for g in gpu_indices)
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.t_mark = None

    def start(self):
        """ONE sampler process (rank 0) for all GPUs of the job, started well before the timed region: nvidia-smi start-up takes NVML /
        driver locks for ~a second and would otherwise stall the first launches of every rank."""
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.gpus}", f"--query-gpu=timestamp,{self.Q}", "--format=csv,noheader,nounits", "-lms", os.environ.get("B2_SAMPLER_MS", "20")],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark(self):
        """samples before this wall-clock instant are outside the timed region and are dropped"""
        import datetime
        self.t_mark = datetime.datetime.now()

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.p.terminate()
        try:
            self.p.wait(2)
        except Exception:
            self.p.kill()
        self.f.flush()
        import datetime
        sm, smax, reasons = [], [], set()
        for line in open(self.f.name):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f")
                if self.t_mark is not None and ts < self.t_mark:
                    continue
                sm.append(float(c[2]))
                smax.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Threads the CPU leg may really use: min(affinity mask, cgroup CPU quota) -- oversubscribing a quota-limited container
    makes OpenMP crawl."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    env = os.environ.get("B2_CPU_THREADS")
    return max(1, int(env)) if env else n


def cpu_reference_leg(args, steps, warmup, budget_s=150.0):
    """The reference's CPU path restated (oracle port) on the host cores: same step, same inputs.  K timed steps after W warm-up steps as asked;
    when that would not finish within `budget_s`, every step processes a bounded SAMPLE of the scan (its first rows), and says so."""
    from oracle import pyoracle as po
    from rmcl_b200 import synth
    po.set_num_threads(host_threads())
    V, F = synth.building(args.faces)
    sc = po.Scene(V, F)
    m = synth.c2_sensor()
    o, d = po.model_rays(m)
    Tsb, Tgt, I = synth.scenario_tsb(), synth.building_gt_pose(), synth.make_transform()
    ranges = synth.noisy_ranges(sc.simulate(Tgt, Tsb, o, d, m.range_max)["ranges"], m.range_max)
    dp, dm, _ = po.dataset_from_ranges(o, d, ranges, m.range_min, m.range_max)
    Tom = rank_pose(synth, 0)

    def step(nr):
        sc.micp_correct_once(o, d[:nr], m.range_max, dp[:nr], dm[:nr], Tom, I, Tsb, ITERATIONS, MAX_DIST, ADAPTIVE_MIN, 0.0, f64_accum=2)

    t0 = time.perf_counter()
    step(m.size)                                  # calibration (also the first warm-up step)
    t_full = time.perf_counter() - t0
    rows = m.phi_size
    if t_full * (steps + warmup) > budget_s:
        rows = max(1, int(m.phi_size * budget_s / (t_full * (steps + warmup))))
    nr = rows * m.theta_size
    for _ in range(max(0, warmup - 1)):
        step(nr)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(nr)
    dt = (time.perf_counter() - t0) / steps
    sample = f"{steps} steps x {nr} of the {m.size} rays of the C2 scan ({rows} of {m.phi_size} rows) + 5 reductions each"
    return nr / dt, dt, host_threads(), nr, sample


_JSON_OUT = None


def pin_to_gpu_numa_node(local_rank):
    """One process per GPU: keep the rank's host threads (launches, the completion-flag spin) on the CPUs next to its GPU.  Without it
    the ~100 us steps of some ranks pay cross-socket latency on every launch and every poll of the mapped completion flag."""
    try:
        import pynvml
        pynvml.nvmlInit()
        hdl = pynvml.nvmlDeviceGetHandleByIndex(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
        words = pynvml.nvmlDeviceGetCpuAffinity(hdl, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, x in enumerate(words) for b in range(64) if (int(x) >> b) & 1}
        allowed = cpus & os.sched_getaffinity(0)
        if len(allowed) >= 2:
            os.sched_setaffinity(0, allowed)
    except Exception:
        pass


def emit(line):
    """The ONE JSON line goes to the process's original stdout; everything else printed during the run (NCCL banners, library chatter)
    was diverted to stderr by main()."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    args = parse()
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)                                   # fd 1 -> stderr for the rest of the run (C libraries included)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": "C2: MICP-L correctOnce, 1 pose x 128x1024 spherical scan, building mesh", "n_faces": args.faces, "rays_per_step_per_gpu": 131072,
              "inner_iterations": ITERATIONS, "poses_per_gpu": 1, "parallelism": f"pose-shard x{world} (map replicated, no collective)",
              "l2": "flushed between timed steps (256 MiB write)", "map_build": "device LBVH (B2_BUILD_MODE=0 selects the host SAH build)",
              "pose": "every step corrects a different pose estimate: the scenario pose with a fresh offset N(1 cm) / N(0.1 deg yaw) per step, like consecutive "
                      "corrections of a tracking filter (B2_BENCH_JITTER=0: the same pose every step); the find kernel orders its tiles by the previous step's warp durations"}

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = max(1, args.steps), max(1, args.warmup)
        val, dt, cores, n, sample = cpu_reference_leg(args, steps, warmup)
        line = {"impl": "reference", "metric": "ray-correspondences/sec", "value": val, "unit": "rays/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "micp_iters_per_s": 1.0 / dt,
                "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "label": "oracle_port_baseline: the repo's own CPU restatement (oracle/), not Embree / rmagine",
                                 "sample": sample + " on the CPU oracle port, OpenMP over rays and over reduction chunks, threads = min(CPU affinity, cgroup CPU quota); Embree/rmagine not buildable here",
                                 "host_logical_cpus": os.cpu_count()},
                "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import rmcl_b200
    from rmcl_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        pin_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.current_stream()
    sampler = ClockSampler(range(world)) if rank == 0 else None
    if sampler:
        sampler.start()

    # ---- set-up (untimed): map build (host SAH -> HBM), model, synthetic scan produced by the library itself at T_gt ----
    V, F = synth.building(args.faces)
    gmap = rmcl_b200.Map(V, F, device=local_rank)
    info = gmap.info()
    m = synth.c2_sensor()
    Tsb, Tgt, I = synth.scenario_tsb(), synth.building_gt_pose(), synth.make_transform()
    h = rmcl_b200.RCCB200Spherical(gmap)
    h.setStream(stream.cuda_stream)
    h.setTsb(Tsb)
    h.setModel(m)
    h.setParams(MAX_DIST, ADAPTIVE_MIN)
    h.find(Tgt)
    ranges = synth.noisy_ranges(h.modelView()["ranges"], m.range_max)
    ranges_pinned = torch.from_numpy(ranges.copy()).pin_memory()
    h.setRanges(ranges)
    Tom = rank_pose(synth, rank)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident steps ----
    # The step is enqueued asynchronously (b2_rcc_correct_once_async) and collected up to QUEUE steps later, so the GPU always has the next
    # steps queued: the CUDA-event interval of a step then contains its kernels only, no host launch / poll latency (with 8 ranks and a clock
    # sampler sharing one host, a single descheduled rank thread used to add milliseconds to one of 20 steps).  Every step is still a complete
    # correctOnce whose result lands in host memory; the synchronous call is what `e2e` times below.
    QUEUE = 4
    # one pose estimate per step (see config["pose"])
    jit = np.random.default_rng(1234 + rank)
    n_pose = args.steps + args.warmup + 8
    Toms = synth.transforms(n_pose)
    for k in range(n_pose):
        if os.environ.get("B2_BENCH_JITTER", "1") != "0":
            Toms[k] = synth.compose(Tom, synth.make_transform(tuple(jit.normal(0.0, 0.01, 3)), (0.0, 0.0, float(jit.normal(0.0, np.radians(0.1))))))
        else:
            Toms[k] = Tom
    for k in range(args.warmup):
        flush.fill_(1)
        h.correctOnce(Toms[k], I, ITERATIONS, 0.0)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    if sampler:
        sampler.mark()
    launches0 = rmcl_b200.kernel_launch_count()
    inflight = 0
    for k, (a, b) in enumerate(ev):
        flush.fill_(2)                      # untimed L2 flush
        a.record(stream)
        h.correctOnceAsync(Toms[args.warmup + k], I, ITERATIONS, 0.0)      # the production kernels: no instrumentation inside the call
        b.record(stream)
        inflight += 1
        if inflight == QUEUE:
            Tn, Td, Cm = h.correctOnceWait()
            inflight -= 1
    while inflight:
        Tn, Td, Cm = h.correctOnceWait()
        inflight -= 1
    launches = rmcl_b200.kernel_launch_count() - launches0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"Tom_new": Tn, "T_onew_oold": Td, "C_merged": Cm})
    step_ms = np.array([a.elapsed_time(b) for a, b in ev], np.float64)
    dev_ms = float(step_ms.sum())

    # ---- the same steps once more with the library's CUDA events around each kernel (stage split; the event records between the two
    #      kernels cost ~3 us per step and keep the second kernel from launching early, hence not inside the timed region above) ----
    h.enableTiming(True)
    find_ms, red_ms = [], []
    for k in range(min(args.steps, 50)):
        flush.fill_(2)
        h.correctOnce(Toms[args.warmup + k], I, ITERATIONS, 0.0)
        f_ms, r_ms = h.lastTiming()
        find_ms.append(f_ms)
        red_ms.append(r_ms)
    h.enableTiming(False)

    # ---- the dominant kernel alone (k_rcc_find at the same pose, L2 flushed): duration for the roofline entry.  Inside the step the find
    #      runs as phase 0 of the fused cooperative kernel, whose total is reported as stage_ms.fused_kernel ----
    Tbm_guess = synth.compose(Tom, I)
    find_alone = []
    for i in range(23):
        flush.fill_(6)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        h.find(Tbm_guess)
        b.record(stream)
        torch.cuda.synchronize()
        if i >= 3:
            find_alone.append(a.elapsed_time(b))

    # ---- end-to-end steps: host ranges in, host result out ----
    for k in range(max(3, args.warmup // 4)):
        h.correctOnce(Toms[k], I, ITERATIONS, 0.0, ranges=ranges_pinned)
    barrier()
    e2e_ms = np.zeros(args.steps)
    for k in range(args.steps):
        flush.fill_(3)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        Tn2, Td2, Cm2 = h.correctOnce(Toms[args.warmup + k], I, ITERATIONS, 0.0, ranges=ranges_pinned)
        e2e_ms[k] = (time.perf_counter() - t0) * 1e3
    e2e_s = float(e2e_ms.sum()) * 1e-3
    barrier()
    # the same call with a PAGEABLE host scan (cudaMemcpyAsync + unpack kernel on a side stream instead of the zero-copy read)
    pg_ms = np.zeros(min(args.steps, 100))
    for k in range(len(pg_ms) + 3):
        flush.fill_(3)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h.correctOnce(Toms[k], I, ITERATIONS, 0.0, ranges=ranges)
        if k >= 3:
            pg_ms[k - 3] = (time.perf_counter() - t0) * 1e3
    barrier()
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max = float(t[0]), float(t[1])
    # per-rank distribution of the per-step device times (p50 / p99 / max per rank): a stall on one rank is visible here, not averaged away
    mine = torch.tensor([np.percentile(step_ms, 50), np.percentile(step_ms, 99), step_ms.max(), step_ms.sum(), np.percentile(e2e_ms, 50), e2e_ms.max()], dtype=torch.float64, device="cuda")
    allr = [torch.zeros_like(mine) for _ in range(world)]
    if dist is not None:
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    per_rank = [{"rank": r, "p50_ms": float(x[0]), "p99_ms": float(x[1]), "max_ms": float(x[2]), "sum_ms": float(x[3]), "e2e_p50_ms": float(x[4]), "e2e_max_ms": float(x[5])} for r, x in enumerate(allr)]
    rays_total = float(m.size) * args.steps * world
    value = rays_total / (dev_ms_max * 1e-3)
    e2e_value = rays_total / (e2e_ms_max * 1e-3)

    # ---- secondary workloads (reported under "extra"; same timing rules) ----
    extra = {}
    if not args.no_extra:
        try:
            extra = extra_workloads(torch, rmcl_b200, synth, gmap, h, m, Tsb, Tgt, stream, flush, dist, world, rank, args)
        except Exception as e:                     # never lose the headline because a secondary workload failed
            extra = {"error": repr(e)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (k_rcc_find).  Live: the kernel's duration (CUDA events, L2 flushed), the L2 / HBM read bandwidth of
    #      this box (the library's micro-benchmark), the SM clock under load.  From the committed ncu capture of the same kernel on the same
    #      input (profiles/counters.json): warp instructions, L1 wavefronts, L2 and DRAM bytes per launch.  Every roof is a time the kernel
    #      cannot beat; frac = that time / measured time; the largest one is the binding roof. ----
    q = np.asarray(synth.compose(Tom, Tsb)["R"], np.float64)
    tsm = np.asarray(synth.compose(Tom, Tsb)["t"], np.float32)
    dirs_s = spherical_dirs_np(m)
    dirs_m = synth._qrot(q[None, :], dirs_s.astype(np.float64)).astype(np.float32)
    vn, vt = gmap.traversal_stats(np.tile(tsm, (len(dirs_m), 1)), dirs_m, m.range_max)
    b_io = 12 + 33                                   # direction table in, point+normal+hit+face+range out
    bytes_per_ray = vn * 224.0 + vt * 48.0 + b_io
    find_s = float(np.mean(find_alone)) * 1e-3
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
    f_sm = ((clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))) * 1e6
    try:
        l2_gbs = rmcl_b200.api.read_bandwidth(32 << 20, 40, local_rank)          # 32 MiB working set: L2-resident
        hbm_read_gbs = rmcl_b200.api.read_bandwidth(4 << 30, 4, local_rank)       # 4 GiB working set: HBM
    except Exception:
        l2_gbs, hbm_read_gbs = None, None
    counters = {}
    try:
        counters = json.load(open(os.path.join(ROOT, "profiles", "counters.json")))
    except Exception:
        pass
    roofline = kernel_roofs("k_rcc_find", f"k_rcc_find#{(m.size + 63) // 64}", find_s, counters, n_sm, f_sm, l2_gbs, hbm_peak, algorithmic_bytes=bytes_per_ray * m.size)
    roofline.update({"peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                     "bytes_per_ray": bytes_per_ray, "nodes_per_ray": vn, "tris_per_ray": vt, "node_bytes": 224, "tri_bytes": 48, "io_bytes_per_ray": b_io,
                     "kernel_ms": find_s * 1e3, "kernel_share_of_step": float(np.mean(find_ms)) / float(np.mean(find_ms) + np.mean(red_ms)),
                     "kernel_rays_per_s": m.size / find_s, "l2_read_gbs_measured": l2_gbs, "hbm_read_gbs_measured": hbm_read_gbs, "sm_mhz_used": f_sm / 1e6,
                     "note": "the 85 MB map stays resident in the 126 MB L2, so HBM does not bind this kernel: `frac_hbm_dram` is the DRAM side, `frac_hbm_algorithmic` the "
                             "contract's algorithmic-bytes figure (can exceed 1 because the bytes come from L1/L2); the binding roof is named in `bound`"})
    loop_s = float(np.mean(red_ms)) * 1e-3
    roof_loop = kernel_roofs("k_icp_loop", f"k_icp_loop<0>#{min(n_sm, (m.size + 511) // 512)}", loop_s, counters, n_sm, f_sm, l2_gbs, hbm_peak, algorithmic_bytes=m.size * 38.0)
    roof_loop["note"] = "five serial grid-wide reductions: latency-bound by construction; algorithmic bytes = one pass over the 38-byte pairs (later passes read registers)"

    def roofs_for(prefix, seconds, alg_bytes):
        keys = [k for k in (counters.get("kernels") or {}) if k.startswith(prefix + "#")]
        key = max(keys, key=lambda k: counters["kernels"][k].get("warp_instructions", 0)) if keys else prefix
        return kernel_roofs(prefix, key, seconds, counters, n_sm, f_sm, l2_gbs, hbm_peak, algorithmic_bytes=alg_bytes)
    if isinstance(extra.get("c3_pf"), dict):
        extra["c3_pf"]["roofline"] = roofs_for("k_pf_update<0>", extra["c3_pf"]["ms_per_step"] * 1e-3, None)
    if isinstance(extra.get("v1_batch"), dict):
        extra["v1_batch"]["roofline"] = roofs_for("k_rcc_fused_batch", extra["v1_batch"]["ms_per_step"] * 1e-3, None)
    if isinstance(extra.get("c4_pinhole"), dict):
        c4 = extra["c4_pinhole"]
        c4["roofline_find"] = kernel_roofs("k_rcc_find", f"k_rcc_find#{(640 * 480 + 63) // 64}", c4["find_alone_ms"] * 1e-3, counters, n_sm, f_sm, l2_gbs, hbm_peak,
                                           algorithmic_bytes=c4["bytes_per_ray"] * 640 * 480)

    # ---- CPU baseline (oracle port) on this box's host cores, bounded sample ----
    cpu = None                                   # N = 1 only: at N > 1 the other ranks' processes share the host cores with it
    if world == 1:
        try:
            val, dt, cores, _, sample = cpu_reference_leg(args, 10, 1, budget_s=30.0)
            cpu = {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "label": "oracle_port_baseline: the repo's own CPU restatement (oracle/), not Embree / rmagine",
                   "sample": sample + " on the CPU oracle port (FP32 merges, OpenMP over rays and reduction chunks); Embree/rmagine unavailable",
                   "ms_per_step": dt * 1e3}
        except Exception as e:
            cpu = {"error": repr(e)}

    line = {"metric": "ray-correspondences/sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "micp_iters_per_s": args.steps * world / (dev_ms_max * 1e-3),
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": int(ranges.nbytes + 1216), "d2h_bytes_per_step": 176,
                    "ms_per_step": e2e_ms_max / args.steps, "timer": "host wall clock around the synchronous C-ABI call, pinned host scan (read zero-copy by the kernel)",
                    "pageable_scan_ms_per_step": float(np.mean(pg_ms)), "pageable_scan_rays_per_s": m.size / (float(np.mean(pg_ms)) * 1e-3)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_icp_loop": roof_loop, "cpu_baseline": cpu,
            "step_ms_per_rank": per_rank, "queue_depth": QUEUE,
            "stage_ms": {"fused_kernel_or_find": float(np.mean(find_ms)), "separate_reduce_launches": float(np.mean(red_ms)), "find_alone": find_s * 1e3},
            "map": {"n_nodes": info["n_nodes"], "bvh_mb": info["bvh_bytes"] / 1e6, "build_ms": info["build_ms"], "max_depth": info["max_depth"], "build_mode": info["build_mode"]},
            "result_check": {"n_meas": int(Cm["n_meas"]), "dt_norm": float(np.linalg.norm(Td["t"]))},
            "extra": extra}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def kernel_roofs(name, key, seconds, counters, n_sm, f_sm, l2_gbs, hbm_gbs, algorithmic_bytes=None):
    """Lower bounds of a kernel's duration from its per-launch counters (profiles/counters.json, ncu) against this box's peaks, as fractions of
    the measured duration.  Returns the contract's roofline object for the binding roof plus every individual roof under `roofs`."""
    c = (counters.get("kernels") or {}).get(key)
    roofs = {}
    if c:
        if c.get("warp_instructions"):
            roofs["issue"] = {"achieved": c["warp_instructions"] / seconds / 1e9, "peak": n_sm * 4 * f_sm / 1e9, "unit": "G warp-inst/s", "per_launch": c["warp_instructions"]}
        if c.get("l1_lsu_wavefronts"):
            roofs["l1_wavefronts"] = {"achieved": c["l1_lsu_wavefronts"] / seconds / 1e9, "peak": n_sm * f_sm / 1e9, "unit": "G wavefronts/s", "per_launch": c["l1_lsu_wavefronts"]}
        if c.get("l2_bytes") and l2_gbs:
            roofs["l2"] = {"achieved": c["l2_bytes"] / seconds / 1e9, "peak": l2_gbs, "unit": "GB/s", "per_launch": c["l2_bytes"]}
        if c.get("dram_bytes") is not None:
            roofs["hbm_dram"] = {"achieved": c["dram_bytes"] / seconds / 1e9, "peak": hbm_gbs, "unit": "GB/s", "per_launch": c["dram_bytes"]}
    if algorithmic_bytes:
        roofs["hbm_algorithmic"] = {"achieved": algorithmic_bytes / seconds / 1e9, "peak": hbm_gbs, "unit": "GB/s", "per_launch": algorithmic_bytes}
    for r in roofs.values():
        r["frac"] = r["achieved"] / r["peak"]
    binding = [k for k in ("issue", "l1_wavefronts", "l2", "hbm_dram") if k in roofs]
    bound = max(binding, key=lambda k: roofs[k]["frac"]) if binding else "hbm_algorithmic"
    top = roofs.get(bound, {"achieved": None, "peak": None, "unit": None, "frac": None})
    out = {"bound": bound, "kernel": name, "achieved": top["achieved"], "peak": top["peak"], "unit": top["unit"], "frac": top["frac"],
           "traffic": (c or {}).get("dram_bytes"), "roofs": roofs, "counters_key": key, "counters_found": bool(c),
           "frac_hbm_dram": roofs.get("hbm_dram", {}).get("frac"), "frac_hbm_algorithmic": roofs.get("hbm_algorithmic", {}).get("frac"),
           "lanes_active_per_instruction": (c or {}).get("lanes_active_per_instruction"), "duration_us": seconds * 1e6,
           "duration_us_under_ncu": (c or {}).get("duration_us_under_ncu")}
    return out


def spherical_dirs_np(m):
    phi = (np.float32(m.phi_min) + np.arange(m.phi_size, dtype=np.float32) * np.float32(m.phi_inc))
    th = (np.float32(m.theta_min) + np.arange(m.theta_size, dtype=np.float32) * np.float32(m.theta_inc))
    cp, sp = np.cos(phi)[:, None], np.sin(phi)[:, None]
    d = np.stack([cp * np.cos(th)[None, :], cp * np.sin(th)[None, :], np.repeat(sp, len(th), 1)], -1)
    return d.reshape(-1, 3).astype(np.float32)


def extra_workloads(torch, rmcl_b200, synth, gmap, h, m, Tsb, Tgt, stream, flush, dist, world, rank, args=None):
    """C3: particle filter 100k particles x 180 beams per GPU (particles sharded across ranks); v1: batched correct(), 1000 poses x vlp16_900."""
    out = {}

    def maxr(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    # ---- C3 ----
    pts = h.modelView()["points"]                       # last find was at the guess pose; any finite scan works as beam source
    beams = synth.pf_beams(pts, 180)
    n_part = 100_000
    P, A = synth.pf_particles(n_part * world)
    from rmcl_b200.shard import shard_range
    b, e = shard_range(len(P), rank, world)
    Pd = torch.from_numpy(P[b:e].view(np.float32).reshape(-1, 8).copy()).cuda()
    A0 = torch.from_numpy(A[b:e].view(np.float32).reshape(-1, 9).copy()).cuda()
    up = rmcl_b200.PCDSensorUpdaterB200(gmap)
    up.setStream(stream.cuda_stream)
    prm = rmcl_b200.PFParams.defaults()
    steps, warm = 10, 3
    tot = 0.0
    for i in range(warm + steps):
        Ad = A0.clone()
        flush.fill_(4)
        a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        up.update(Pd, Ad, Tsb, beams, prm)
        bb.record(stream)
        torch.cuda.synchronize()
        if i >= warm:
            tot += a.elapsed_time(bb)
    ms = maxr(tot) / steps
    # end to end with host particles
    # pinned host staging (like the scan of the headline step)
    Ph = torch.from_numpy(P[b:e].view(np.uint8).copy()).pin_memory().numpy().view(P.dtype).reshape(-1)
    Ah = torch.from_numpy(A[b:e].view(np.uint8).copy()).pin_memory().numpy().view(A.dtype).reshape(-1)
    A_init = Ah.copy()
    up.update(Ph, Ah, Tsb, beams, prm, inplace=True)               # untimed: first call sizes the staging buffers
    e2e_t = 0.0
    for _ in range(5):
        Ah[:] = A_init                                   # every timed update starts from the same particle attributes
        flush.fill_(4); torch.cuda.synchronize()
        t0 = time.perf_counter()
        up.update(Ph, Ah, Tsb, beams, prm, inplace=True)  # pinned host particles in, updated attributes back in the same (pinned) array
        e2e_t += time.perf_counter() - t0
    e2e = maxr(e2e_t / 5)
    out["c3_pf"] = {"workload": f"C3: particle-filter sensor update, {n_part} particles x 180 beams per GPU, 1M-triangle mesh", "rays_per_s": n_part * world * 180 / (ms * 1e-3),
                    "ms_per_step": ms, "e2e_rays_per_s": n_part * world * 180 / e2e, "e2e_ms_per_step": e2e * 1e3,
                    "h2d_bytes_per_step": n_part * (32 + 36) + 180 * 32, "d2h_bytes_per_step": n_part * 36}
    # ---- the same update for a CONVERGED particle cloud (tracking): the updater times its two ray mappings and keeps the faster one ----
    try:
        rngc = np.random.default_rng(7 + rank)
        Pc = P[b:e].copy()
        gt = synth.building_gt_pose()
        Pc["t"][:, 0] = gt["t"][0] + rngc.normal(0, 0.3, len(Pc)); Pc["t"][:, 1] = gt["t"][1] + rngc.normal(0, 0.3, len(Pc)); Pc["t"][:, 2] = gt["t"][2]
        yawc = rngc.normal(0.0, np.radians(5.0), len(Pc))
        Pc["R"][:, 0] = 0; Pc["R"][:, 1] = 0; Pc["R"][:, 2] = np.sin(yawc / 2); Pc["R"][:, 3] = np.cos(yawc / 2)
        Pcd = torch.from_numpy(Pc.view(np.float32).reshape(-1, 8).copy()).cuda()
        res = {}
        for mode in (0, 3):
            up.setMapping(mode)
            tot = 0.0
            for i in range(4 + 6):
                Ad = A0.clone()
                flush.fill_(4)
                a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                up.update(Pcd, Ad, Tsb, beams, prm)
                bb.record(stream)
                torch.cuda.synchronize()
                if i >= 4:
                    tot += a.elapsed_time(bb)
            res[mode] = maxr(tot) / 6
        out["c3_pf_tracking"] = {"workload": f"C3 for a converged cloud: {n_part} particles per GPU within sigma 0.3 m / 5 deg of one pose, 180 beams",
                                 "ms_per_step_lanes_are_beams": res[0], "ms_per_step": res[3], "rays_per_s": n_part * world * 180 / (res[3] * 1e-3),
                                 "mapping_chosen": up.mapping()[1], "note": "mapping 2 = lanes are particles sorted by (heading, cell) on the device; the sort is inside the timed step"}
        up.setMapping(3)
    except Exception as ex:
        out["c3_pf_tracking"] = {"error": repr(ex)}
    # ---- C5 (BASELINE.json configs[4]): 1M particles x 360 beams sharded 8 ways = 125 000 x 360 per GPU; runs when 8 ranks are present
    #      (B2_BENCH_C5=1 forces the per-GPU share on fewer GPUs)
    if world == 8 or os.environ.get("B2_BENCH_C5") == "1":
        beams5 = synth.pf_beams(pts, 360)
        P5, A5 = synth.pf_particles(125_000 * world, seed=7)
        b5, e5 = shard_range(len(P5), rank, world)
        P5d = torch.from_numpy(P5[b5:e5].view(np.float32).reshape(-1, 8).copy()).cuda()
        A50 = torch.from_numpy(A5[b5:e5].view(np.float32).reshape(-1, 9).copy()).cuda()
        tot5 = 0.0
        for i in range(2 + 5):
            A5d = A50.clone()
            flush.fill_(4)
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            up.update(P5d, A5d, Tsb, beams5, prm)
            bb.record(stream)
            torch.cuda.synchronize()
            if i >= 2:
                tot5 += a.elapsed_time(bb)
        ms5 = maxr(tot5) / 5
        out["c5_pf"] = {"workload": f"C5: particle-filter sensor update, {125_000 * world} particles x {len(beams5)} beams over {world} GPU(s), 1M-triangle mesh",
                        "rays_per_s": 125_000 * world * len(beams5) / (ms5 * 1e-3), "ms_per_step": ms5}
    # ---- the whole particle-filter cycle on the device (SURVEY 8f2): motion -> sensor update -> stats (8-byte all-reduce) -> Gladiator
    # resampling (all-gather of the particle set when sharded); particles never leave HBM
    glad = rmcl_b200.GladiatorConfig.defaults()
    Tmo = synth.make_transform((0.02, 0.0, 0.0), (0.0, 0.0, 0.01))
    # sharded resampling: opponents over NVLink peer memory (CUDA IPC: 4-byte likelihood reads, 68-byte records for winners only); all-gather
    # of the whole particle set as the fallback when the GPUs cannot map each other's memory
    exchange, p2p_bytes, variants_equal = "none", None, None
    if world > 1:
        try:
            up.p2pConnect(dist, n_part)
            exchange = "p2p"
        except Exception as ex:                      # noqa: BLE001
            exchange = f"allgather (p2p unavailable: {ex})"
    Pc, Ac = Pd.clone(), A0.clone()
    tot = 0.0
    for i in range(warm + steps):
        flush.fill_(4)
        a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        up.motionUpdate(Pc, Ac, Tmo, 0.01)
        up.update(Pc, Ac, Tsb, beams, prm)
        up.likelihoodStats(Ac, dist if world > 1 else None)
        if world > 1 and exchange == "p2p":
            Pn, An, p2p_bytes = up.resampleShardedP2P(Pc, Ac, dist, glad, seed=1234, step=i, want_traffic=True)
        elif world > 1:
            Pn, An = up.resampleSharded(Pc, Ac, dist, glad, seed=1234, step=i)
        else:
            Pn, An = torch.empty_like(Pc), torch.empty_like(Ac)
            up.resample(Pc, Ac, Pn, An, glad, seed=1234, step=i)
        bb.record(stream)
        torch.cuda.synchronize()
        if i == warm + steps - 1 and world > 1 and exchange == "p2p":          # correctness on hardware: both exchange variants give the same particles
            Pg, Ag = up.resampleSharded(Pc, Ac, dist, glad, seed=1234, step=i)
            torch.cuda.synchronize()
            ok = torch.tensor([int(torch.equal(Pg, Pn) and torch.equal(Ag, An))], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            variants_equal = bool(int(ok[0]))
        Pc, Ac = Pn, An
        if i >= warm:
            tot += a.elapsed_time(bb)
    ms_cycle = maxr(tot) / steps
    out["c3_pf_cycle"] = {"workload": f"C3 full cycle on the device: motion + sensor update ({n_part} particles x 180 beams per GPU) + stats + Gladiator resampling",
                          "rays_per_s": n_part * world * 180 / (ms_cycle * 1e-3), "ms_per_cycle": ms_cycle,
                          "exchange": "none" if world == 1 else exchange,
                          "exchange_bytes_per_rank_per_cycle": None if world == 1 else ({"p2p_read": p2p_bytes, "allgather_would_receive": (world - 1) * n_part * 68} if exchange == "p2p"
                                                                                          else {"allgather_received": (world - 1) * n_part * 68}),
                          "p2p_equals_allgather": variants_equal}
    # ---- v1 batched correct ----
    hv = rmcl_b200.SphereCorrectorB200(gmap)
    hv.setStream(stream.cuda_stream)
    hv.setTsb(Tsb)
    mv = synth.vlp16_900()
    mv.range_min = 0.0
    hv.setModel(mv)
    hv.setParams(1.0, 0.15)
    hv.find(Tgt)
    hv.setInputData(hv.modelView()["ranges"])
    n_poses = 1000
    T = synth.transforms(n_poses)
    T[:] = synth.compose(Tgt, synth.scenario_pose_offset())
    rng = np.random.default_rng(rank)
    T["t"] += rng.uniform(-0.05, 0.05, (n_poses, 3)).astype(np.float32)
    Td_ = torch.from_numpy(T.view(np.float32).reshape(-1, 8).copy()).cuda()
    tot = 0.0
    for i in range(warm + steps):
        flush.fill_(5)
        a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        hv.correct(Td_)
        bb.record(stream)
        torch.cuda.synchronize()
        if i >= warm:
            tot += a.elapsed_time(bb)
    ms = maxr(tot) / steps
    out["v1_batch"] = {"workload": "v1 correct(): 1000 poses x vlp16_900 (14400 rays) per GPU, fused trace+P2L+Umeyama", "rays_per_s": n_poses * world * mv.size / (ms * 1e-3),
                       "ms_per_step": ms, "reference_numbers": "Embree 0.201 s, OptiX 0.0169 s per correct() on a 1M-face sphere (BASELINE.md)"}
    # ---- closest-point correspondences (SURVEY 8f3) on the C2 scan: CPCEmbree::find + the same inner iterations ----
    ds = h.datasetView()
    hc = rmcl_b200.CPCB200(gmap)
    hc.setStream(stream.cuda_stream)
    hc.setTsb(Tsb); hc.setParams(MAX_DIST, ADAPTIVE_MIN); hc.setDataset(ds["points"], ds["mask"])
    Tomc = synth.compose(Tgt, synth.scenario_pose_offset())
    Ic = synth.make_transform()
    cpc = {}
    for name, skip in (("reference_behaviour", False), ("skip_masked", True)):
        hc.setOptions(skip_masked=skip)
        tt = []
        for i in range(13):
            flush.fill_(8)
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); hc.find(Tomc); bb.record(stream)
            torch.cuda.synchronize()
            if i >= 3:
                tt.append(a.elapsed_time(bb))
        cpc[name] = {"find_ms": maxr(float(np.mean(tt))), "queries_per_s": m.size * world / (maxr(float(np.mean(tt))) * 1e-3)}
    out["cpc_c2"] = {"workload": "closest-point correspondences (CPCB200::find) for the 131072 dataset points of the C2 scan, 1M-triangle building", **cpc,
                     "note": "reference_behaviour queries every dataset point like CPCEmbree.cpp:30-43; skip_masked leaves out the 2 % masked-out points (dropped beams far outside the map) whose results no statistic uses"}
    # ---- C4 (BASELINE.json configs[3]): PinholeCorrector, 640 x 480 depth camera on the 500k-triangle indoor mesh ----
    if rank == 0 or world > 1:
        V4, F4 = synth.indoor(500_000)
        map4 = rmcl_b200.Map(V4, F4, device=torch.cuda.current_device())
        m4 = synth.c4_sensor()
        h4 = rmcl_b200.RCCB200Pinhole(map4)
        h4.setStream(stream.cuda_stream)
        h4.setTsb(Tsb); h4.setModel(m4); h4.setParams(1.0, 0.15)
        T4 = synth.indoor_gt_pose()
        h4.find(T4)
        r4 = synth.noisy_ranges(h4.modelView()["ranges"], m4.range_max)
        h4.setRanges(r4)
        r4_pinned = torch.from_numpy(r4.copy()).pin_memory()
        Tom4 = synth.compose(T4, synth.scenario_pose_offset())
        I4 = synth.make_transform()
        n4, warm4 = 40, 5
        for _ in range(warm4):
            flush.fill_(7); h4.correctOnce(Tom4, I4, ITERATIONS, 0.0)
        ev4 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n4)]
        infl = 0
        for a, bb in ev4:
            flush.fill_(7)
            a.record(stream); h4.correctOnceAsync(Tom4, I4, ITERATIONS, 0.0); bb.record(stream)
            infl += 1
            if infl == 4:
                out4 = h4.correctOnceWait(); infl -= 1
        while infl:
            out4 = h4.correctOnceWait(); infl -= 1
        torch.cuda.synchronize()
        ms4 = maxr(sum(a.elapsed_time(bb) for a, bb in ev4)) / n4
        f4 = []
        for i in range(13):
            flush.fill_(7)
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); h4.find(synth.compose(Tom4, I4)); bb.record(stream)
            torch.cuda.synchronize()
            if i >= 3:
                f4.append(a.elapsed_time(bb))
        e4 = 0.0
        for i in range(n4 + 3):
            flush.fill_(7); torch.cuda.synchronize()
            t0 = time.perf_counter()
            h4.correctOnce(Tom4, I4, ITERATIONS, 0.0, ranges=r4_pinned)
            if i >= 3:
                e4 += time.perf_counter() - t0
        e4 = maxr(e4) / n4
        from rmcl_b200.api import _PinholeModel  # noqa: F401
        px = ((np.arange(m4.width, dtype=np.float32) - np.float32(m4.cx)) / np.float32(m4.fx))[None, :].repeat(m4.height, 0)
        py = ((np.arange(m4.height, dtype=np.float32) - np.float32(m4.cy)) / np.float32(m4.fy))[:, None].repeat(m4.width, 1)
        nrm = np.sqrt(px * px + py * py + 1.0)
        d4 = np.stack([1.0 / nrm, -px / nrm, -py / nrm], -1).reshape(-1, 3).astype(np.float32)
        Tsm4 = synth.compose(Tom4, Tsb)
        d4m = synth._qrot(np.asarray(Tsm4["R"], np.float64)[None, :], d4.astype(np.float64)).astype(np.float32)
        vn4, vt4 = map4.traversal_stats(np.tile(np.asarray(Tsm4["t"], np.float32), (len(d4m), 1)), d4m, m4.range_max)
        out["c4_pinhole"] = {"workload": "C4: PinholeCorrector correctOnce, 1 pose x 640x480 depth image, 500k-triangle indoor mesh (find + 5 inner iterations)",
                             "rays_per_s": m4.size * world / (ms4 * 1e-3), "ms_per_step": ms4, "find_alone_ms": float(np.mean(f4)), "find_rays_per_s": m4.size / (float(np.mean(f4)) * 1e-3),
                             "e2e_rays_per_s": m4.size * world / e4, "e2e_ms_per_step": e4 * 1e3, "h2d_bytes_per_step": int(r4.nbytes + 1216), "d2h_bytes_per_step": 176,
                             "nodes_per_ray": vn4, "tris_per_ray": vt4, "bytes_per_ray": vn4 * 224.0 + vt4 * 48.0 + 45, "n_meas": int(out4[2]["n_meas"]),
                             "pairs_per_loop_thread": "2 in registers + 3 in shared memory (307 200 pairs on 148 x 512 threads)"}
    return out


if __name__ == "__main__":
    main()
