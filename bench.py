#!/usr/bin/env python
"""bench.py -- keyframe-window optimize() throughput (BASELINE.json metric) on N B200s.

A "step" = one pass of the hot path over one batch: Estimator::optimize(10 iterations) on every
resident 10-keyframe / 2000-landmark stereo window (BASELINE.json configs[1]; synthetic, seeded).
  value : iterations/s (accepted + rejected dogleg iterations, as Ceres counts them) with the windows
          already resident in HBM, timed with CUDA events on the library's stream, max over ranks.
  e2e   : the same metric through the C-ABI with HOST buffers: okb_window_upload (H2D) +
          okb_optimize + okb_window_download (D2H) inside the timed region.
  roofline / cpu_baseline : see DESIGN.md "Measurement".
`--impl reference` times the CPU oracle (the restated okvis_ceres path; the real reference cannot be
built here) on the box's host cores on the same workload.
Windows shard across ranks with no data-path collective (independent windows): weak scaling.
"""
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

METRIC = "keyframe-window optimize() iters/sec (10KF/2k-lm stereo)"
ITERS = 10


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.stop_flag = threading.Event()
        self.sm, self.sm_max, self.reasons = [], [], set()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.sm.append(float(out[0]))
                self.sm_max.append(float(out[1]))
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=3)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.sm_max)), "reasons": sorted(self.reasons)}


def fp64_roofline(achieved_gflops):
    """The Jacobian / J^T J / Schur group against the FP64 peak (the bound that really applies: ~50 FLOP per byte).  The
    driver's MEASURED_PEAKS.json has no FP64 figure; the peak is this project's own measurement (tools/fp64_peak.cu,
    DFMA and DMMA both 37 TFLOP/s on this B200), committed under profiles/."""
    path = os.path.join(ROOT, "profiles", "r01_fp64_peak.json")
    try:
        pk = json.load(open(path))
        peak = 1e3 * float(max(pk["fp64_fma_tflops"], pk["fp64_dmma_tflops"]))
        src = "profiles/r01_fp64_peak.json (tools/fp64_peak.cu)"
    except Exception:
        peak, src = 37000.0, "fallback 37 TFLOP/s"
    return {"bound": "fp64", "achieved": achieved_gflops, "peak": peak, "unit": "GFLOP/s", "frac": achieved_gflops / peak,
            "flops": "SURVEY 8d model: 1500 N_obs + 324 sum f_l^2 + d^3/3 + 14000 (K-1) per window-iteration", "peak_source": src}


def make_windows(n_distinct, base_idx):
    from okvis_b200 import synthetic
    return [synthetic.make_window(2, base_idx + i) for i in range(n_distinct)]


def host_cpus():
    """CPUs this process may really use: os.cpu_count() capped by the affinity mask and the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p_ = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(round(q / p_))))
        except (OSError, ValueError):
            pass
    return n


def cpu_oracle_pass(windows, n_win, threads):
    """One bounded CPU sample: n_win cfg-2 windows, each solved by one oracle thread (optimize(ITERS) + the
    landmark-quality pass of Estimator::optimize), `threads` windows in flight.  Building the problems (the
    reference's addObservation bookkeeping) is not part of optimize() and stays outside the timed region.
    Returns (iterations, seconds)."""
    from oracle import oracle_py as op
    from concurrent.futures import ThreadPoolExecutor
    probs = [op.OracleProblem(windows[i % len(windows)]) for i in range(n_win)]

    def solve_one(p):
        s = p.solve(ITERS, 1)
        p.state(with_quality=True)
        return s["iterations"]

    with ThreadPoolExecutor(max_workers=threads) as ex:
        t0 = time.perf_counter()
        it = sum(ex.map(solve_one, probs))
        dt = time.perf_counter() - t0
    for p in probs:
        p.close()
    return it, dt


def run_reference(args):
    """CPU arm: the oracle (restated reference path) on the host cores, all threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cpus()
    windows = make_windows(8, 0)
    # warm-up doubles as the choice of the thread count: the usable CPUs (cgroup quota, affinity) and a little
    # oversubscription are tried and the fastest configuration is kept
    best_t, best_rate = cores, 0.0
    cand = sorted({cores, 2 * cores, max(1, cores // 2)}, reverse=True)
    for wstep in range(max(args.warmup, len(cand))):
        t_ = cand[wstep % len(cand)]
        it, dt = cpu_oracle_pass(windows, 2 * t_, t_)
        if it / dt > best_rate:
            best_rate, best_t = it / dt, t_
    n_win = 2 * best_t
    times, iters = [], 0
    for step in range(args.steps):
        it, dt = cpu_oracle_pass(windows, n_win, best_t)
        times.append(dt)
        iters += it
    cores = best_t
    total = sum(times)
    value = iters / total
    w = windows[0]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "iterations/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg-2: 10-keyframe stereo (2x752x480), 2000 landmarks, 200 Hz IMU window, optimize(10)",
                   "windows_per_step": n_win, "n_obs": int(len(w.obs)), "iterations_per_optimize": ITERS},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores, "kind": "port",
                         "sample": "%d windows x optimize(%d) per step, one oracle thread per window" % (n_win, ITERS)},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "restated-reference CPU path (oracle/): the original Ceres/SuiteSparse binary cannot be built here",
    }
    print(json.dumps(line))


def reference_matcher_us(A, B, threads=4, reps=5):
    """Host time of the REFERENCE's DenseMatcher::match (oracle/_ref/libokvis_matcher_ref.so: okvis_matcher's own sources,
    oracle/Makefile.ref) on two descriptor lists with the frontend's 4 matcher threads (Frontend.cpp:80); None if the
    library did not travel.  Test-infrastructure code on the cpu_baseline side of the bench only."""
    import ctypes as C
    so = os.path.join(ROOT, "oracle", "_ref", "libokvis_matcher_ref.so")
    if not os.path.exists(so) or len(A) == 0 or len(B) == 0:
        return None
    try:
        lib = C.CDLL(so)
        A = np.ascontiguousarray(A, np.uint8)
        B = np.ascontiguousarray(B, np.uint8)
        oa, od = np.zeros(len(B), np.int32), np.zeros(len(B), np.float32)
        args = (C.c_void_p(A.ctypes.data), len(A), C.c_void_p(B.ctypes.data), len(B), A.shape[1], C.c_float(60.0), 4, threads,
                C.c_void_p(oa.ctypes.data), C.c_void_p(od.ctypes.data))
        lib.okr_match_hamming(*args)
        t0 = time.perf_counter()
        for _ in range(reps):
            lib.okr_match_hamming(*args)
        return (time.perf_counter() - t0) * 1e6 / reps
    except Exception:
        return None


def frontend_leg(ctx, cam, rank=0, world=1, with_cpu=True):
    """Secondary measurement (north_star rows S-V, BASELINE.json configs[2]): keypoint detect/describe and the all-pairs
    Hamming matcher through the C-ABI with host buffers (host clock, copies included), next to the CPU oracle on a
    bounded sample.  Two parameter sets: cfg-3 (uniformity radius 15, <= 1000 keypoints on a dense texture, 1000 x 1000
    match) and OKVIS' shipped yaml (radius 40, <= 400).  Images shard over ranks per image (SURVEY 8e row 3): every
    rank works on its own seeded stereo pair; rank 0 reports its own timings, the caller sums images/s over ranks."""
    from okvis_b200 import images
    from oracle import oracle_py as op
    R = np.eye(3)
    out = {"note": "host buffers in/out, host clock; sequential DenseMatcher semantics (top-k lists and assignbest on the device)"}
    seed = 0x0B200 + 3000 + 17 * rank
    dense_l = images.textured_image(seed, n_shapes=2600)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    dense_r = np.roll(dense_l, -12, axis=1).astype(np.float64) + rng.normal(0, 2.0, dense_l.shape)
    dense_r = np.clip(np.rint(dense_r), 0, 255).astype(np.uint8)
    left, right = images.stereo_pair()
    for tag, (il, ir), kw in (("cfg3", (dense_l, dense_r), dict(uniformity_radius=15.0, max_keypoints=1000)),
                              ("production", (left, right), dict(uniformity_radius=40.0, max_keypoints=400))):
        for s_, im in enumerate((il, ir)):
            ctx.detect_describe(im, cam, R, cam_slot=s_, **kw)
        reps = 20
        t0 = time.perf_counter()
        for _ in range(reps):
            kl, dl = ctx.detect_describe(il, cam, R, cam_slot=0, **kw)
            kr, dr = ctx.detect_describe(ir, cam, R, cam_slot=1, **kw)
        dd_ms = (time.perf_counter() - t0) * 1e3 / (2 * reps)
        ctx.hamming_match(dl, dr)
        t0 = time.perf_counter()
        for _ in range(50):
            ctx.hamming_match(dl, dr)
        m_us = (time.perf_counter() - t0) * 1e6 / 50
        o = {"detect_describe_ms_per_image": dd_ms, "keypoints": [int(len(kl)), int(len(kr))], "hamming_match_us": m_us,
             "hamming_match_shape": [int(len(dl)), int(len(dr))],
             "params": "uniformity radius %.0f px, absolute threshold 800, <= %d keypoints, 48-byte descriptors" % (kw["uniformity_radius"], kw["max_keypoints"]),
             # SURVEY 8d algorithmic traffic: 3.3 MB per image (image + score planes + descriptors), (nA+nB)*48 + nA*32 B per match
             "detect_describe_GBps": 3.3e-3 / (dd_ms * 1e-3), "hamming_Gpairs_per_s": len(dl) * len(dr) / (m_us * 1e-6) / 1e9}
        if with_cpu:
            t0 = time.perf_counter()
            op.detect_describe(il, cam, R, **kw)
            o["cpu_oracle_detect_describe_ms_per_image"] = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            for _ in range(3):
                op.match_hamming(dl, dr)
            o["cpu_oracle_hamming_match_us"] = (time.perf_counter() - t0) * 1e6 / 3
            ref_us = reference_matcher_us(dl, dr)
            if ref_us is not None:       # the reference's own DenseMatcher (oracle/_ref, okvis_matcher compiled unmodified), 4 matcher threads
                o["cpu_reference_hamming_match_us"] = ref_us
        out[tag] = o
    rng = np.random.Generator(np.random.PCG64(5))
    A = rng.integers(0, 256, (1000, 48), dtype=np.uint8)
    Bm = A[rng.permutation(1000)].copy()
    Bm[:, :4] ^= rng.integers(0, 256, (1000, 4), dtype=np.uint8)
    ctx.hamming_match(A, Bm)
    t0 = time.perf_counter()
    for _ in range(50):
        ctx.hamming_match(A, Bm)
    out["hamming_1000x1000_us"] = (time.perf_counter() - t0) * 1e6 / 50
    A = rng.integers(0, 256, (8192, 48), dtype=np.uint8)
    Bm = rng.integers(0, 256, (8192, 48), dtype=np.uint8)
    ctx.hamming_match(A, Bm, threshold=200.0)
    t0 = time.perf_counter()
    for _ in range(5):
        ctx.hamming_match(A, Bm, threshold=200.0)
    out["hamming_8192x8192_gcmp_per_s"] = 8192.0 * 8192.0 / ((time.perf_counter() - t0) / 5) / 1e9
    out["images_per_s_this_gpu"] = 1e3 / out["cfg3"]["detect_describe_ms_per_image"]
    return out


def pin_to_gpu_numa(gpu_index):
    """Pins this process (and the host threads it starts later) to the CPUs of the NUMA node the GPU hangs off, so that
    the command packing and the pinned staging buffers of a rank stay local to its GPU.  Returns the node or None."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        dom, rest = bus.split(":", 1)
        node = int(open("/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:], rest)).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def latency_leg(torch, dev, local_rank, window, reps=20):
    """B = 1 latency (SURVEY 8d): ONE resident cfg-2 window, reset + optimize(10) + quality pass, CUDA events on the
    library stream, plus the host wall time of the blocking okb_optimize call (launch + sync + summary read-back)."""
    from okvis_b200 import capi
    c1 = capi.Context(local_rank, 1)
    try:
        c1.upload(0, window)
        stream = torch.cuda.ExternalStream(c1.stream, device=dev)
        dev_ms, wall_ms, iters = [], [], 0
        for rep in range(reps + 3):
            c1.reset(0, 1)
            torch.cuda.synchronize(dev)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                ev0.record(stream)
                c1.optimize_async(0, 1, max_iterations=ITERS)
                ev1.record(stream)
            s = c1.optimize_finish(0, 1)[0]
            t1 = time.perf_counter()
            torch.cuda.synchronize(dev)
            if rep >= 3:
                dev_ms.append(ev0.elapsed_time(ev1))
                wall_ms.append((t1 - t0) * 1e3)
                iters = s["iterations"]
        return {"latency_b1_ms": float(np.median(dev_ms)), "latency_b1_wall_ms": float(np.median(wall_ms)),
                "latency_b1_min_ms": float(min(dev_ms)), "iterations": int(iters), "reps": reps,
                "what": "one resident cfg-2 window: optimize(%d) + landmark-quality pass, device time (CUDA events) and host wall time of the blocking call" % ITERS}
    finally:
        c1.close()


def cfg5_leg(torch, dist, dev, rank, world, local_rank, reps=5):
    """BASELINE.json configs[4]: ONE 20-keyframe / 4-camera / 8000-landmark window, landmarks sharded lm_idx % world over
    the ranks, partial reduced systems all-reduced through NVLink peer-memory mailboxes inside the solver kernels
    (okb_shard_*).  Times reset + optimize(10) with CUDA events on the library stream, max over ranks.  At world = 1
    this is the unsharded single-GPU latency the speed-up at 2/4/8 GPUs refers to."""
    from okvis_b200 import capi, sharding, synthetic
    w = synthetic.make_window(5, 0)
    c5 = capi.Context(local_rank, 1)
    try:
        if world > 1:
            sharding.connect_shards(c5, dist, dev, rank, world, len(w.poses))
            sw, _ = sharding.shard_window(w, rank, world)
        else:
            sw = w
        c5.upload(0, sw)
        stream = torch.cuda.ExternalStream(c5.stream, device=dev)

        def sync():
            torch.cuda.synchronize(dev)
            if dist is not None:
                dist.barrier()
                torch.cuda.synchronize(dev)

        times, iters, wait_us, rounds = [], 0, 0.0, 0
        for rep in range(reps + 2):
            sync()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                ev0.record(stream)
                c5.reset(0, 1)
                c5.optimize_async(0, 1, max_iterations=ITERS)
                ev1.record(stream)
            s = c5.optimize_finish(0, 1)[0]
            torch.cuda.synchronize(dev)
            if rep >= 2:
                times.append(ev0.elapsed_time(ev1))
                iters += s["iterations"]
                if world > 1:
                    st = c5.shard_stats(0)
                    wait_us += st["wait_us"]
                    rounds += st["rounds"]
        t = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        return {"workload": "cfg-5: single 20-keyframe 4-camera window, 8000 landmarks, %d observations, optimize(%d)" % (len(w.obs), ITERS),
                "world": world, "partition": "lm_idx % world, dense blocks replicated, reduced solve redundant",
                "collective": "sum of the (6K+1)^2 Schur accumulator + pose blocks over peer-memory mailboxes (NVLink stores + flags), fused into k_shard_push / k_solve; second 8-scalar exchange inside k_solve",
                "ms_per_optimize": total_ms / reps, "iterations_per_s": iters / (total_ms * 1e-3), "iterations": iters // reps,
                "final_cost": s["final_cost"], "termination": s["termination"],
                "exchange_wait_us_per_round": (wait_us / rounds) if rounds else None, "reps": reps}
    finally:
        c5.close()


DUMP_BYTES = 64 << 20
SUMMARY_FIELDS = ("initial_cost", "final_cost", "iterations", "num_successful_steps", "termination", "imu_redo_count",
                  "final_radius")


def dump_outputs(out_dir, ctx, summaries, budget=DUMP_BYTES, suffix=""):
    """What the last timed step handed its caller: the estimates of every window (poses, speed/bias, landmarks, landmark
    quality) and the solver summaries (solve_time_s left out: it is a host timing), one float64 .npy per array.  When
    all windows exceed `budget` bytes, a fixed seeded sample of windows is written; window_index.npy says which."""
    n = len(summaries)
    per_window = sum(v.nbytes for v in ctx.download(0).values()) + 8 * (len(SUMMARY_FIELDS) + 1)
    keep = n if n * per_window <= budget else max(1, budget // per_window)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).permutation(n)[:keep])
    states = [ctx.download(int(i)) for i in idx]
    arrays = {k: np.stack([s[k] for s in states]) for k in ("poses", "speed_bias", "landmarks", "quality")}
    arrays.update({k: np.array([summaries[i][k] for i in idx], np.float64) for k in SUMMARY_FIELDS})
    arrays["window_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + suffix + ".npy"), v.astype(np.float64))


def run_b200(args):
    import torch
    from okvis_b200 import capi
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = pin_to_gpu_numa(local_rank)
    B = args.batch
    Be = max(1, min(B, args.e2e_batch))                 # windows per slot range of the e2e leg (two ranges alternate)
    ctx = capi.Context(local_rank, max(B, 2 * Be))
    # independent windows: global window w runs on rank w mod world (SURVEY 8e), no data-path collective
    from okvis_b200 import sharding, synthetic
    windows = [synthetic.make_window(2, w) for w in sharding.shard_indices(world * args.distinct, world, rank)]
    ctx.upload_batch(0, [windows[i % len(windows)] for i in range(B)], args.host_threads)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step():
        ctx.reset(0, B)
        return ctx.optimize(0, B, max_iterations=ITERS)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches
    ctx.profile_enable(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 0
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            last = step()
            iters += sum(s["iterations"] for s in last)
        ev1.record(stream)
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    launches = ctx.kernel_launches - launches0
    clocks = sampler.result() if rank == 0 else None
    if args.dump_outputs:       # before the e2e leg reuses these slots
        dump_outputs(args.dump_outputs, ctx, last, DUMP_BYTES // world, "" if world == 1 else "_rank%d" % rank)

    # ---- e2e through the C-ABI with HOST buffers, resident windows (SURVEY 8f-3): the windows live on the device; every
    # step the host restores a slot to its uploaded estimates (okb_window_reset, device side), drops the newest frame
    # and adds it again -- pose, speed/bias, the ImuError term with its samples and that frame's observations, i.e. what
    # Estimator::addStates + addObservation send per camera frame -- then optimizes and downloads ALL estimates
    # (poses, speed/bias, landmarks, quality).  Each step therefore solves the same graph as the resident leg from the
    # same initial estimates.  Two slot ranges alternate so that the host-side command packing, the H2D copy, the
    # device-side graph compile and the D2H copy of one range overlap the solve of the other (transfer stream).
    e2e_steps = max(12, 2 * args.steps)     # the two-range pipeline needs a fill and a drain step: amortised like in a long stream
    range_windows = [windows[i % len(windows)] for i in range(Be)]
    descs = ctx.make_descs(range_windows)              # descriptors only point at the host arrays
    for base in (0, Be):
        for i, w_ in enumerate(range_windows):
            ctx.reserve(base + i, len(w_.poses), len(w_.landmarks), len(w_.obs) + 4096, len(w_.imu_samples) + 256)
        ctx.upload_batch(base, range_windows, args.host_threads, descs)
    full_upload_bytes = sum(ctx.h2d_bytes(i) for i in range(Be))
    host_out = {base: ctx.alloc_outputs(base, Be) for base in (0, Be)}   # host result buffers, reused every step
    prepared = {base: [ctx.prepare_readd_newest(base + i, w_) for i, w_ in enumerate(range_windows)] for base in (0, Be)}
    d2h_range = sum(v.nbytes for o in host_out[0][0] for v in o.values()) + Be * 48   # estimates + summaries
    h2d_seen = []

    def upload_range(base):
        ctx.reset(base, Be)                 # device side: estimates as uploaded (no host traffic)
        ctx.readd_newest(prepared[base])    # host side: command appends into the pinned per-slot buffers
        ctx.commit(base, Be)                # one H2D copy per slot + device-side interpreter / compile
        if not h2d_seen:
            h2d_seen.append(sum(ctx.h2d_bytes(base + i) for i in range(Be)))   # counted by the library per commit
        return h2d_seen[0]

    def download_range(base):
        ctx.download_batch(base, Be, host_out[base])
        return d2h_range

    def e2e_run(n_steps):
        # software pipeline over two window ranges: while the device optimizes range `cur`, the host downloads
        # the estimates of the previous step and sends the next step's frame (transfer stream)
        it = 0
        h2d = d2h = 0
        h2d += upload_range(0)
        pending = None
        for st in range(n_steps):
            base = (st % 2) * Be
            ctx.optimize_async(base, Be, max_iterations=ITERS)
            if pending is not None:
                d2h += download_range(pending)
            if st + 1 < n_steps:
                h2d += upload_range(((st + 1) % 2) * Be)
            ss = ctx.optimize_finish(base, Be)
            it += sum(x["iterations"] for x in ss)
            pending = base
        d2h += download_range(pending)
        return it, h2d / n_steps, d2h / n_steps

    e2e_run(2)
    barrier()
    t_host = time.perf_counter()
    e_iters, h2d, d2h = e2e_run(e2e_steps)
    torch.cuda.synchronize(dev)
    e2e_wall = time.perf_counter() - t_host     # host packing is part of the end-to-end path
    barrier()
    (elapsed_ms, e2e_ms), (iters_all, e_iters_all, launches_all) = sharding.reduce_measurement(
        dist, dev, [elapsed_ms, e2e_wall * 1e3], [iters, e_iters, launches])
    launches_all = int(launches_all)
    try:        # secondary leg, all ranks take part (collective set-up); must not break the headline
        cfg5_res = cfg5_leg(torch, dist, dev, rank, world, local_rank)
    except Exception as e:
        cfg5_res = {"error": repr(e)}

    lat = None
    if rank == 0:
        try:
            lat = latency_leg(torch, dev, local_rank, windows[0])
        except Exception as e:
            lat = {"error": repr(e)}
    try:        # frontend leg on every rank: images shard per image, no collective (SURVEY 8e row 3)
        frontend = frontend_leg(ctx, windows[0].cameras[0], rank, world, with_cpu=(rank == 0))
        ips = frontend["images_per_s_this_gpu"]
    except Exception as e:       # the headline measurement must not depend on this leg
        frontend, ips = {"error": repr(e)}, 0.0
    (_,), (ips_all,) = sharding.reduce_measurement(dist, dev, [0.0], [ips])
    if isinstance(frontend, dict):
        frontend["images_per_s_all_gpus"] = ips_all
    if rank == 0:
        peak, peak_kind = load_peaks()
        w = windows[0]
        bytes_iter = float(np.mean([x.algorithmic_bytes_per_iteration() for x in windows]))
        flops_iter = float(np.mean([x.algorithmic_flops_per_iteration() for x in windows]))
        # kernel A ("Jacobian + JtJ/Schur build"): one launch processes one linearisation of all B windows
        lm_ms = prof["landmarks_ms"] / max(prof["landmarks_launches"], 1)
        sv_ms = prof["solve_ms"] / max(prof["solve_launches"], 1)
        achieved = B * bytes_iter / (lm_ms * 1e-3) / 1e9
        total_k = prof["landmarks_ms"] + prof["solve_ms"] + prof["quality_ms"]
        # DRAM bytes per launch of the group from the committed ncu --set full captures (profiles/), scaled to B
        traffic, traffic_src = None, None
        import glob
        tpaths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
        tpath = tpaths[-1] if tpaths else ""
        if tpath:
            tj = json.load(open(tpath))
            ks = tj.get("kernels", {})
            if all(k in ks for k in ("k_linearize", "k_lmblock", "k_schur")):
                traffic = sum(ks[k]["dram_read_bytes"] + ks[k]["dram_write_bytes"] for k in ("k_linearize", "k_lmblock", "k_schur"))
                traffic = traffic * B / float(tj.get("windows", B))
                traffic_src = "profiles/%s (ncu dram__bytes_read+write.sum of the three kernels at %d windows)" % (os.path.basename(tpath), tj.get("windows", B))
        # CPU baseline: bounded sample of the same workload on this box's host cores -- one oracle thread per
        # window; as many windows in flight as there are usable CPUs (cgroup quota) or twice that, whichever is faster
        cores = host_cpus()
        cpu_iters, cpu_dt, n_cpu = 0, 1.0, 1
        for t_ in ([1] if args.skip_cpu else sorted({cores, 2 * cores}, reverse=True)):
            it_, dt_ = cpu_oracle_pass(windows, t_, t_)
            if it_ / dt_ > cpu_iters / cpu_dt:
                cpu_iters, cpu_dt, n_cpu = it_, dt_, t_
        cores = n_cpu
        cfg5 = cfg5_res
        line = {
            "metric": METRIC, "value": iters_all / (elapsed_ms * 1e-3), "unit": "iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "cfg-2: 10-keyframe stereo (2x752x480), 2000 landmarks, 200 Hz IMU window, optimize(10)",
                       "windows_per_gpu": B, "n_obs": int(len(w.obs)), "iterations_per_optimize": ITERS,
                       "parallelism": "independent windows, %d per GPU, no collective" % B,
                       "l2": "inputs larger than L2 (%.0f MB resident per GPU)" % (B * 3.0)},
            "e2e": {"value": e_iters_all / (e2e_ms * 1e-3), "unit": "iterations/s", "h2d_bytes_per_step": int(h2d) * world,
                    "d2h_bytes_per_step": int(d2h) * world, "windows_per_gpu": Be, "steps": e2e_steps,
                    "full_window_upload_bytes": int(full_upload_bytes) * world,
                    "note": "resident windows: per step reset (device) + re-add of the newest frame with its IMU term and observations (H2D) "
                            "+ optimize(10) + download of all estimates (D2H); two slot ranges alternate so transfers overlap the solve"},
            "gpu_launches": launches_all,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_linearize + k_lmblock + k_schur (residuals, Jacobian factors, J^T J, Schur complement)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "peak_source": peak_kind, "avg_launch_ms": lm_ms, "algorithmic_bytes_per_window_iteration": bytes_iter,
                         "fp64_gflops": B * flops_iter / (lm_ms * 1e-3) / 1e9,
                         "share_of_kernel_time": prof["landmarks_ms"] / max(total_k, 1e-9),
                         "k_solve_avg_launch_ms": sv_ms, "k_solve_share": prof["solve_ms"] / max(total_k, 1e-9)},
            "roofline_fp64": fp64_roofline(B * flops_iter / (lm_ms * 1e-3) / 1e9),
            "cpu_baseline": {"value": cpu_iters / cpu_dt, "unit": "iterations/s", "cores": cores, "kind": "port",
                             "sample": "%d windows x optimize(%d) + quality pass, one oracle thread per window, %d threads" % (n_cpu, ITERS, cores)},
            "latency": lat,
            "host": {"numa_node": numa_node, "usable_cpus": host_cpus()},
            "frontend": frontend,
            "cfg5_sharded_window": cfg5,
        }
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=592, help="resident windows per GPU (4 per SM)")
    ap.add_argument("--e2e-batch", type=int, default=592, help="windows per step of the e2e leg (two slot ranges of this size alternate)")
    ap.add_argument("--skip-cpu", action="store_true", help="tuning runs only: shrink the cpu_baseline sample to one window")
    ap.add_argument("--host-threads", type=int, default=12, help="host threads packing/uploading windows in the e2e leg")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic windows per rank (replicated to fill the batch)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the estimates and summaries of the last timed step to DIR/<name>.npy (float64, <= 64 MB "
                         "in all) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computed")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
