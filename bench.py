#!/usr/bin/env python
"""bench.py -- headline benchmark of the scan-matching hot path (BASELINE.json: correspondences/s per linearize()).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] -- an IntegratedVGICPFactor with a 1,000,000-point source cloud
linearized against a 0.5 m Gaussian voxel map built from a 1,000,000-point target (synthetic street scene, seeded).
A "step" is ONE linearize(): correspondence search for every source point + reduction into H, b.  A fresh pose
(xi ~ U(+-0.01 rad, +-0.1 m), what LM iterations look like) is used at every step.

  value  : correspondences/s = source points processed by all ranks / max-over-ranks device time (CUDA events), inputs
           resident in HBM, poses on the device, results left on the device.
  e2e    : same metric through the public host API (NonlinearFactorSetGPU.linearize / ShardedFactorSet.linearize):
           per step the poses go host->device and the H, b records come back device->host inside the timed region
           (that is exactly the per-linearize traffic of the reference's NonlinearFactorSetGPU,
           src/gtsam_points/cuda/nonlinear_factor_set_gpu.cpp:91-124; clouds and maps are uploaded once, at construction).
  N > 1  : weak scaling -- every rank owns one such factor (independent factors shard with no data-path collective),
           then ONE all-reduce(sum) over the [N x 128] float64 record buffer publishes all H, b on every rank.
  --impl reference : the reference's CPU algorithm (oracle/liboracle.so, a line-by-line restatement -- the reference
           itself needs GTSAM/Eigen and cannot be built here) on all host cores, same workload and metric.

L2 is flushed between timed steps (256 MiB write followed by a 256 MiB read of other memory, so the cache holds only clean
foreign lines); each step is bracketed by its own CUDA events.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only: nothing is cached next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_SOURCE = 1_000_000
N_TARGET = 1_000_000
RESOLUTION = 0.5
POSE_ROT, POSE_TRANS = 0.01, 0.1
METRIC = "correspondences/s per linearize() (1M-pt VGICP)"
UNIT = "correspondences/s"
WORKLOAD = "IntegratedVGICPFactor: 1M-pt source into 0.5 m GaussianVoxelMap (1M-pt target), one linearize() per step"


def workload_config():
    """`config` is IDENTICAL in both arms (the driver compares them); arm-specific facts go into `detail`."""
    return {
        "workload": WORKLOAD,
        "n_source": N_SOURCE,
        "n_target": N_TARGET,
        "resolution": RESOLUTION,
        "pose_perturbation": {"rot_rad": POSE_ROT, "trans_m": POSE_TRANS},
        "l2": "flushed between timed steps (GPU arm: 256 MiB write then 256 MiB read; CPU arm: working set 320 MB >> LLC)",
    }


AFFINITY = sorted(os.sched_getaffinity(0))  # taken at import: once libgomp binds the main thread, sched_getaffinity(0) shrinks to its place


def pin_openmp_env():
    """SURVEY.md 8d: the CPU arm runs thread-pinned.  libgomp reads these when it is first loaded, so they are set before
    torch / the oracle are imported.  (Explicit user settings win.)"""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_WAIT_POLICY", "active")  # worker threads spin between the timed calls instead of being woken up for each


def host_info():
    info = {"nproc": os.cpu_count(), "affinity": len(AFFINITY), "omp_proc_bind": os.environ.get("OMP_PROC_BIND"), "omp_places": os.environ.get("OMP_PLACES"), "omp_wait_policy": os.environ.get("OMP_WAIT_POLICY")}
    try:
        import psutil

        info["physical_cores"] = psutil.cpu_count(logical=False)
    except Exception:
        pass
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["cpu"] = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


def make_inputs(rank: int):
    from gtsam_points_b200 import synthetic as syn

    tp, tc = syn.make_cloud(N_TARGET, stream=2 * rank + 1)
    sp, sc = syn.make_cloud(N_SOURCE, stream=2 * rank + 2)
    return tp, tc, sp, sc


def make_poses(rank: int, count: int):
    from gtsam_points_b200 import synthetic as syn

    rng = np.random.default_rng(1000 + rank)
    return np.stack([syn.random_pose(rng, POSE_ROT, POSE_TRANS) for _ in range(count)])


def dump_records(out_dir, loop: str, records):
    """Linearized records of a timed loop's last step ([F x >= 122] float64, b2_linearized layout) ->
    out_dir/<loop>_<field>.npy, one float64 array per field with the factor as leading axis."""
    from gtsam_points_b200 import capi

    fields = [capi.unpack_linearized(r) for r in np.atleast_2d(np.asarray(records, dtype=np.float64))]
    os.makedirs(out_dir, exist_ok=True)
    for k in fields[0]:
        np.save(os.path.join(out_dir, f"{loop}_{k}.npy"), np.array([f[k] for f in fields], dtype=np.float64))


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML (~1 kHz; the timed region of this
    benchmark is tens of milliseconds, far below nvidia-smi's sampling period)."""

    def __init__(self, index: int):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            return
        bits = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")

        def loop():
            while not self._stop.is_set():
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = int(get_reasons(h))
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                time.sleep(0.001)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any (profiles/*.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("vgicp_linearize_dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference's OpenMP CPU path, all host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_threads(orc) -> int:
    """One OpenMP thread per PHYSICAL core: the float64 loop does not gain from SMT siblings (measured on the B200 host:
    64 threads on 64 cores 20 M correspondences/s, 128 threads on the same cores 4.3 M/s), and the reference arm must show
    the CPU path at its best."""
    try:
        import psutil

        phys = psutil.cpu_count(logical=False)
        if phys:
            # not clamped by omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to its workers, and the oracle
            # passes the count explicitly (`num_threads(n)` clause), which overrides that default
            return max(1, min(int(phys), len(AFFINITY)))
    except Exception:
        pass
    return max(orc.max_threads(), 1)


def time_cpu(tp, tc, sp, sc, poses, warmup: int, steps: int):
    import oracle_lib as orc

    threads = cpu_threads(orc)
    vm = orc.VoxelMap(RESOLUTION)
    tgt = orc.Cloud(tp, tc)
    vm.insert(tgt)
    src = orc.Cloud(sp, sc)
    f = orc.Factor(vm, src, num_threads=threads)
    for i in range(warmup):
        f.linearize_raw(poses[i % len(poses)])
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        last = f.linearize_raw(poses[(warmup + i) % len(poses)])
        times.append(time.perf_counter() - t0)
    return times, threads, last


def cpu_value(times) -> float:
    """correspondences/s from the MEDIAN call (SURVEY.md 8d: median of >= 10 linearize() calls after warm-up)."""
    return N_SOURCE / float(np.median(times))


def time_cpu_native(steps: int, warmup: int):
    """Same oracle compiled with -march=native ON THIS HOST (the reference's BUILD_WITH_MARCH_NATIVE option, off by default):
    run in a child process because the library handle is process-global.  Returns correspondences/s or None."""
    try:
        with tempfile.TemporaryDirectory(prefix="b2_oracle_native_") as tmp:
            env = dict(os.environ, B2_ORACLE_NATIVE=tmp)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup), "--no-native"],
                                 env=env, capture_output=True, text=True, timeout=600, preexec_fn=lambda: os.sched_setaffinity(0, AFFINITY))
        return float(json.loads(out.stdout.strip().splitlines()[-1])["value"])
    except Exception:
        return None


def time_cpu_single_thread(tp, tc, sp, sc, pose):
    """The reference's DEFAULT is num_threads = 1 (factors/impl/integrated_gicp_factor_impl.hpp:29): one warm-up + one timed
    linearize() of the same workload on one core, reported next to the all-cores number (SURVEY.md 8d)."""
    import oracle_lib as orc

    vm = orc.VoxelMap(RESOLUTION)
    tgt = orc.Cloud(tp, tc)
    vm.insert(tgt)
    f = orc.Factor(vm, orc.Cloud(sp, sc), num_threads=1)
    f.linearize_raw(pose)
    t0 = time.perf_counter()
    f.linearize_raw(pose)
    return N_SOURCE / (time.perf_counter() - t0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    tp, tc, sp, sc = make_inputs(0)
    steps = args.steps
    poses = make_poses(0, steps + args.warmup)
    native = bool(os.environ.get("B2_ORACLE_NATIVE"))
    # the -march=native child runs FIRST: afterwards this process's own OpenMP team exists and (OMP_WAIT_POLICY=active) spins
    # on the cores between parallel regions, which would steal them from the child
    native_value = time_cpu_native(steps, args.warmup) if (not native and not args.no_native) else None
    times, threads, last = time_cpu(tp, tc, sp, sc, poses, args.warmup, steps)
    if args.dump_outputs:
        dump_records(args.dump_outputs, "linearize", last)  # same workload and last pose as the GPU arm's "linearize" loop
    value = cpu_value(times)
    sample = (f"median of {steps} linearize() calls of the full 1M-pt workload after {args.warmup} warm-up, one pinned OpenMP thread per physical core"
              + (", -march=native build" if native else ", reference default flags (-O3, no -march=native)"))
    cpu_baseline = {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "min_ms": 1e3 * float(np.min(times)), "max_ms": 1e3 * float(np.max(times))}
    if native_value is not None:
        cpu_baseline["native_value"] = native_value
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.median(times)),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(),
        "detail": {"threads": threads, "host": host_info()},
        "cpu_baseline": cpu_baseline,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import ctypes as C

    import torch
    import torch.distributed as dist

    import gtsam_points_b200 as g
    from gtsam_points_b200 import capi
    from gtsam_points_b200.distributed import ShardedFactorSet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        try:
            os.sched_setaffinity(0, AFFINITY)  # whatever an inherited OMP_PROC_BIND did to the main thread when libgomp was loaded
        except OSError:
            pass
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner to STDOUT at init when NCCL_DEBUG=VERSION is in the environment; stdout must carry
        # exactly one JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    stream = torch.cuda.Stream(device=dev)
    K, W = args.steps, args.warmup
    dp = C.POINTER(C.c_double)
    L = capi.lib()
    # the -march=native CPU child runs before this process creates its own OpenMP team (parity check / cpu_baseline below): with
    # OMP_WAIT_POLICY=active that team spins on the cores between parallel regions and would steal them from the child
    native_cpu_value = time_cpu_native(10, 2) if (world == 1 and not args.no_cpu_baseline and not args.no_native) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    with torch.cuda.stream(stream):
        ctx = g.Context(local_rank, stream=stream.cuda_stream)
        # L2 flush between timed steps: write 256 MiB (> 126 MB of L2), then stream 256 MiB of other memory through it with
        # reads so that the cache is left full of CLEAN foreign lines -- none of the workload's data is resident, and the timed
        # kernel does not also pay for writing the flush buffer's dirty lines back to DRAM.
        flush_w = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        flush_r = torch.zeros(32 << 20, dtype=torch.int64, device=dev)

        def flush_l2(i):
            if not args.no_flush:
                flush_w.fill_(i & 0xFF)
                flush_r.sum()

        def time_steps(step_fn, poses_c, warmup, steps, rendezvous=None):
            """max-over-ranks device time of `steps` calls of step_fn(pose), L2 flushed before each, own CUDA events per step.
            rendezvous (N > 1): enqueues a device-side rendezvous of the ranks' GPUs, so that the GPUs -- not the python
            processes, whose launch skew is tens of microseconds -- enter each timed step together (the exchange inside a step
            must not absorb another rank's L2 flush or host jitter; everything is enqueued ahead, nothing blocks the host)."""
            for i in range(warmup):
                step_fn(poses_c[i])
            barrier()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for i in range(steps):
                flush_l2(i)
                if world > 1:
                    (rendezvous or barrier)()
                ev[i][0].record(stream)
                step_fn(poses_c[warmup + i])
                ev[i][1].record(stream)
            # drain the device BEFORE the next collective: an NCCL kernel enqueued while persistent one-CTA-per-SM kernels that wait
            # for a peer are still queued can take the SMs those kernels need on one rank and wait for them on the other (deadlock)
            torch.cuda.synchronize(dev)
            barrier()
            ms = np.array([a.elapsed_time(b) for a, b in ev])
            return max_over_ranks(float(ms.sum())), ms

        # ================= headline: one 1M-point factor per rank (weak scaling) =================
        tp, tc, sp, sc = make_inputs(rank)
        poses = make_poses(rank, K + W)
        poses_c = [np.ascontiguousarray(p.reshape(1, 16)) for p in poses]
        poses_p = [p.ctypes.data_as(dp) for p in poses_c]  # argument marshalling is not part of any measured call
        t0 = time.perf_counter()
        vm = g.GaussianVoxelMapGPU(RESOLUTION, ctx)
        vm.insert(g.PointCloud(tp, tc, ctx=ctx, flags=capi.B2_CLOUD_NO_REORDER))
        src = g.PointCloud(sp, sc, ctx=ctx)
        factor = g.IntegratedVGICPFactor(2 * rank, 2 * rank + 1, vm, src, ctx=ctx)
        setup_s = time.perf_counter() - t0
        sset = ShardedFactorSet([factor], [rank], world, ctx=ctx)
        vinfo, cinfo = vm.info(), src.info()
        launches0 = sset.set.launch_count()
        issue_linearize = L.b2_factor_set_issue_linearize

        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        if world == 1:
            # single GPU: the step IS the kernel launch (no exchange).  The asynchronous entry point (NonlinearFactorGPU's
            # issue_linearize): host pose in (by value with the launch), record left on the device
            def dev_step(pose):
                capi.check(issue_linearize(sset.set.h, pose.ctypes.data_as(dp), sset.d_all.data_ptr()))
        else:
            def dev_step(pose):
                sset.linearize_device(pose)  # one launch: linearize + peer stores of the records + in-kernel flag wait
        dev_total_ms, step_ms = time_steps(dev_step, poses_c, W, K, sset.device_barrier)
        # launches of THIS library's kernels inside the timed region: (warm-up + timed) steps launched equally many, the timed share is K of them
        launches_dev = (sset.set.launch_count() - launches0) * K // (K + W)
        rec = sset.d_all.cpu().numpy().copy()
        exchange_path = "peer stores in the kernel epilogue (NVLink) + in-kernel flag wait (b2_exchange, CUDA IPC)" if sset.exchange is not None else "ONE all-reduce of [N x 128] f64 (NCCL)"
        if world > 1 and sset.exchange is not None:
            # untimed cross-check: the fused peer-memory exchange must deliver exactly what the all-reduce path delivers
            saved, sset.exchange = sset.exchange, None
            sset.d_all = torch.zeros((sset.num_global, capi.B2_LINEARIZED_DOUBLES), dtype=torch.float64, device=dev)
            sset.d_deltas.copy_(torch.as_tensor(poses_c[-1], device=dev))
            ref_all = sset.linearize_device().clone()
            barrier()
            sset.exchange = saved
            got_all = sset.linearize_device(poses_c[-1]).clone()
            barrier()
            assert torch.equal(ref_all, got_all), "peer-memory exchange and all-reduce disagree"
        n_inliers = int(rec[rank, 121])
        if world == 1:
            kern_ms = step_ms
        else:  # kernel-only timing for the roofline (same launch, no exchange)
            def kern_step(pose):
                capi.check(issue_linearize(sset.set.h, pose.ctypes.data_as(dp), sset.d_local.data_ptr()))
            _, kern_ms = time_steps(kern_step, poses_c, 1, K, sset.device_barrier)
        kern_ms_mean = max_over_ranks(float(kern_ms.mean()))

        # ---- end-to-end arm: the public host entry point with HOST buffers (poses in, H/b records out) ----
        # N = 1: the C-ABI call itself (b2_factor_set_linearize), which is what NonlinearFactorSetGPU.linearize and the C++
        #        adapters issue; N > 1: ShardedFactorSet.linearize (host poses -> kernel + exchange -> host records).
        h_out = np.zeros((1, capi.B2_LINEARIZED_DOUBLES))
        linearize_host = L.b2_factor_set_linearize
        h_out_p = h_out.ctypes.data_as(dp)

        def e2e_step(pose, pose_p):
            if world == 1:
                capi.check(linearize_host(sset.set.h, pose_p, h_out_p))  # the C-ABI call a C++ caller makes: host pose in, host record out
                return h_out
            return sset.linearize(pose)

        for i in range(W):
            e2e_step(poses_c[i], poses_p[i])
        barrier()
        e2e_s = 0.0
        for i in range(K):
            flush_l2(i)
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            out = e2e_step(poses_c[W + i], poses_p[W + i])
            e2e_s += time.perf_counter() - t0
        e2e_rec = np.array(out, copy=True)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        e2e_ms = max_over_ranks(e2e_s * 1e3)

        # ================= sub-record: STRONG scaling -- the same 1M-point factor split over the ranks (SURVEY 8e(2)) =================
        # every rank holds the whole target map and a contiguous 1/N slice of rank 0's source cloud; the N partial records are
        # exchanged like any other records and summed (H, b and the error are sums over points)
        strong = strong_rec = None
        if world > 1 and not args.no_extra:
            tp0, tc0, sp0, sc0 = make_inputs(0)
            vm0 = g.GaussianVoxelMapGPU(RESOLUTION, ctx)
            vm0.insert(g.PointCloud(tp0, tc0, ctx=ctx, flags=capi.B2_CLOUD_NO_REORDER))
            lo, hi = rank * N_SOURCE // world, (rank + 1) * N_SOURCE // world
            part = g.IntegratedVGICPFactor(0, 1, vm0, g.PointCloud(sp0[lo:hi], sc0[lo:hi], ctx=ctx), ctx=ctx)
            ss = ShardedFactorSet([part], [rank], world, ctx=ctx)
            poses0 = [np.ascontiguousarray(p.reshape(1, 16)) for p in make_poses(0, K + W)]
            total = {}

            def strong_step(pose):
                total["rec"] = ss.linearize_device(pose).sum(0)  # the factor's H, b, error = sum of the ranks' partial records

            ms_total, strong_ms = time_steps(strong_step, poses0, W, K, ss.device_barrier)
            strong_rec = total["rec"].cpu().numpy()
            strong = {"workload": "ONE 1M-pt VGICP factor, source points split over the ranks, partial H/b records summed", "scaling": "strong",
                      "ms_per_step": ms_total / K, "step_ms_min_median_max": [float(strong_ms.min()), float(np.median(strong_ms)), float(strong_ms.max())], "value": N_SOURCE * K / (ms_total * 1e-3), "unit": UNIT, "inliers": int(total["rec"][121].item())}
            del ss, part, vm0

        # ================= sub-record: cfg4 share -- 32 factors x 200k points per GPU in ONE set (256 factors at 8 GPUs) =================
        cfg4 = None
        if not args.no_extra:
            F4, N4 = 32, 200_000
            from gtsam_points_b200 import synthetic as syn

            t0 = time.perf_counter()
            fs, keep = [], []
            for i in range(F4):
                gid = rank * F4 + i
                tpi, tci = syn.make_cloud(N4, stream=2 * gid + 1, scene_seed=2000 + gid // 4)
                spi, sci = syn.make_cloud(N4, stream=2 * gid + 2, scene_seed=2000 + gid // 4)
                vmi = g.GaussianVoxelMapGPU(RESOLUTION, ctx)
                vmi.insert(g.PointCloud(tpi, tci, ctx=ctx, flags=capi.B2_CLOUD_NO_REORDER))
                fs.append(g.IntegratedVGICPFactor(2 * gid, 2 * gid + 1, vmi, g.PointCloud(spi, sci, ctx=ctx), ctx=ctx))
                keep.append(vmi)
            setup4_s = time.perf_counter() - t0
            s4 = ShardedFactorSet(fs, list(range(rank * F4, (rank + 1) * F4)), world * F4, ctx=ctx)
            rng4 = np.random.default_rng(4000 + rank)
            poses4 = [np.ascontiguousarray(np.stack([syn.random_pose(rng4, POSE_ROT, POSE_TRANS) for _ in range(F4)]).reshape(F4, 16)) for _ in range(K + W)]
            if world == 1:
                issue = L.b2_factor_set_issue_linearize

                def cfg4_step(pose):
                    capi.check(issue(s4.set.h, pose.ctypes.data_as(dp), s4.d_all.data_ptr()))
            else:
                def cfg4_step(pose):
                    s4.linearize_device(pose)
            ms_total, _ = time_steps(cfg4_step, poses4, W, K, s4.device_barrier)
            rec4 = s4.d_all.cpu().numpy()
            cfg4 = {"workload": f"ISAM2-style relinearize: {F4} VGICP factors x {N4} points per GPU in ONE launch ({world * F4} factors sharded over {world} GPU(s)), records exchanged",
                    "scaling": "weak", "factors_per_gpu": F4, "points_per_factor": N4, "ms_per_step": ms_total / K, "value": world * F4 * N4 * K / (ms_total * 1e-3), "unit": UNIT,
                    "hit_rate": float(rec4[:, 121].sum() / (world * F4 * N4)), "setup_s": setup4_s}

    if rank == 0:
        value = world * N_SOURCE * K / (dev_total_ms * 1e-3)
        e2e_value = world * N_SOURCE * K / (e2e_ms * 1e-3)
        peak, peak_src = measured_hbm_peak()
        V, NB = int(vinfo.num_voxels), int(vinfo.num_buckets)
        # ALGORITHMIC bytes per launch (SURVEY.md 8d): compact reference layout, every distinct input byte once:
        # N (12 + 36) + N_buckets 16 + V (12 + 36 + 4) + 992.  N_buckets is counted for the REFERENCE's table (power of two,
        # load <= 0.5: 16-byte VoxelBucket, types/gaussian_voxelmap_gpu.hpp:30-33), not for this library's sparser one
        # (load <= 0.25, `num_buckets` below), so that table slack does not inflate the achieved figure.
        NB_alg = 1 << max(14, (2 * V - 1).bit_length())
        alg_bytes = N_SOURCE * (12 + 36) + NB_alg * 16 + V * (12 + 36 + 4) + 992
        achieved = alg_bytes / (kern_ms_mean * 1e-3) / 1e9
        # ---- untimed parity check of the headline workload against the CPU oracle (rank 0; indices bit-exact, H / b 1e-9) ----
        # (runs AFTER every timed loop: with OMP_WAIT_POLICY=active -- as the CPU arm wants it at N = 1 -- the oracle's OpenMP team keeps
        # spinning on all cores afterwards and would compete with the host threads of the end-to-end loop)
        parity = None
        if rank == 0 and not args.no_cpu_baseline:
            import oracle_lib as orc

            ovm = orc.VoxelMap(RESOLUTION)
            ovm.insert(orc.Cloud(tp, tc))
            of = orc.Factor(ovm, orc.Cloud(sp, sc), num_threads=cpu_threads(orc))
            ref = of.linearize_raw(poses[-1])
            h_chk = np.zeros((1, capi.B2_LINEARIZED_DOUBLES))
            capi.check(L.b2_factor_set_linearize(sset.set.h, poses_p[-1], h_chk.ctypes.data_as(dp)))
            corr_equal = bool(np.array_equal(factor.correspondences(), of.correspondences()))
            rel = float(np.abs(h_chk[0, :121] - ref[:121]).max() / np.abs(ref[:121]).max())
            parity = {"checked_against": "CPU oracle, same cloud and pose", "correspondences_identical": corr_equal, "inliers": int(h_chk[0, 121]),
                      "oracle_inliers": int(ref[121]), "max_rel_err_H_b_error": rel}
            assert corr_equal and int(h_chk[0, 121]) == int(ref[121]) and rel < 1e-9, parity

        if args.dump_outputs:
            dump_records(args.dump_outputs, "linearize", rec)
            dump_records(args.dump_outputs, "linearize_host", e2e_rec)
            if strong_rec is not None:
                dump_records(args.dump_outputs, "strong_scaling", strong_rec)
            if cfg4 is not None:
                dump_records(args.dump_outputs, "cfg4", rec4)

        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cs, cw = 10, 2
            times, threads, _ = time_cpu(tp, tc, sp, sc, poses, cw, cs)
            cpu_baseline = {
                "value": cpu_value(times),
                "unit": UNIT,
                "cores": threads,
                "kind": "port",
                "sample": f"median of {cs} linearize() calls of the full 1M-pt workload after {cw} warm-up, one pinned OpenMP thread per physical core, reference default flags",
                "min_ms": 1e3 * float(np.min(times)),
                "max_ms": 1e3 * float(np.max(times)),
                "native_value": native_cpu_value,  # same code, -march=native (the reference's optional BUILD_WITH_MARCH_NATIVE); timed first
                "host": host_info(),
                "single_thread_value": time_cpu_single_thread(tp, tc, sp, sc, poses[0]),  # the reference's default num_threads = 1
            }
        line = {
            "metric": METRIC,
            "value": value,
            "unit": UNIT,
            "n_gpus": world,
            "steps": K,
            "warmup": W,
            "ms_per_step": dev_total_ms / K,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(),
            "detail": {
                "num_voxels": V,
                "num_buckets": NB,
                "inliers": n_inliers,
                "hit_rate": n_inliers / N_SOURCE,
                "factors_per_gpu": 1,
                "parallelism": f"factor-sharded x{world}" + (f"; records exchanged by {exchange_path}" if world > 1 else ""),
                "source_storage": {"point_bytes": int(cinfo.point_bytes), "cov_bytes": int(cinfo.cov_bytes), "morton_ordered": bool(cinfo.reordered)},
                "l2_flush": not args.no_flush,
                "setup_s": setup_s,
                "parity_check": parity,
                "e2e_minus_kernel_us": 1e3 * (e2e_ms / K - kern_ms_mean),
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 128 * 1, "d2h_bytes_per_step": 1024 * world, "ms_per_step": e2e_ms / K},
            "gpu_launches": int(launches_dev),
            "roofline": {
                "bound": "hbm",
                "achieved": achieved,
                "peak": peak,
                "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": ncu_traffic(),
                "kernel": "b2::ws::factor_kernel<float,double,VGICP,LINEARIZE,SINGLE> (by-value pose)",
                "kernel_ms": kern_ms_mean,
                "algorithmic_bytes_per_launch": alg_bytes,
                "algorithmic_bytes_formula": "N*48 + N_buckets_ref*16 + V*52 + 992 with N_buckets_ref = 2^ceil(log2(2V)) (>= 16384)",
                "peak_source": peak_src,
            },
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "extra": {"strong_scaling_1m_factor": strong, "cfg4_share": cfg4},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed linearize() calls of every measured loop")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sub-records (strong-scaling split, cfg4 share): headline numbers only")
    ap.add_argument("--no-native", action="store_true", help="reference arm: skip the secondary -march=native measurement")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic only: keep L2 warm between steps (NOT a valid bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the H, b, error and inlier count that the last timed step of each timed loop computed to DIR/<loop>_<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    # Thread pinning is for the process that times the CPU oracle: the reference arm, or the single-process CUDA arm (cpu_baseline).
    # NOT for the ranks of a multi-GPU run: with OMP_PROC_BIND set, libgomp binds every process's MAIN thread to the first place
    # when it is loaded, i.e. all ranks to the same core -- two ranks still fit its two hardware threads, eight take turns in
    # scheduler quanta (measured: 31 ms per end-to-end step at 8 ranks, 92 us at 2).
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" or world == 1:
        pin_openmp_env()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
