#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path: forward 3-D C2C FFT, GFlops/s = 5 N^3 log2(N^3) / t
(3dmpifft_opt/fftSpeed3d_c2c.cpp:126-128), per-stage t0..t3 ms, HBM-roofline fraction.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl dfft|reference] [--size 512] [--precision double]
                    [--dump-outputs DIR]

A "step" is one forward transform of the synthetic N^3 cube (BASELINE.json configs[1]: 512^3 double on
1 GPU; the same cube sharded over N GPUs = strong scaling).  N > 1 runs one process per GPU under
torchrun; torch.distributed is plumbing only (bootstrap of IPC handles, barrier, max-over-ranks).

`--impl reference` times the reference tree's own CPU FFT on the host cores: heFFTe 2.1.0 with its `stock` backend
(oracle/_ref/libheffte_ref.so, built from /root/reference/heffte/heffteBenchmark by oracle/ref_heffte/Makefile; slab
decomposition, p2p_plined reshape like heffteSpeed.sh), one rank per physical core, ranks pinned.  The reference's GPU hot
path (3dmpifft_opt) needs HIP/hiprtc/rocFFT/MPI and cannot be built here (DESIGN.md).  If the prebuilt library is missing the
arm falls back to the OpenMP oracle port (oracle/oracle_fft.c) and says so (`kind: "port"`).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only; nothing is cached in it
# the CPUs this process may use, taken BEFORE any OpenMP runtime (torch's) binds the main thread to one core
try:
    CPUS_ALLOWED = sorted(os.sched_getaffinity(0))
except AttributeError:
    CPUS_ALLOWED = list(range(os.cpu_count() or 1))


def pin_openmp_threads():
    """CPU legs only: OpenMP threads bound to cores, one per place.  Must run before the OpenMP runtime in question starts (the
    oracle's libgomp), and must NOT be set for the GPU arm's processes: under torchrun every rank's main thread would be bound to
    the first place -- the same core -- and the ranks' kernel launches would time-share it (measured: 512^3 on 4 GPUs 1.88 ms per
    step host-bound against 0.87 ms of device time, profiles/r2_final_bench_n4_hostbound.json)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")


DUMP_BYTES = 32 << 20   # --dump-outputs: data written per run, over all ranks


def dump_output(directory, name, out, count, ranks):
    """Writes the first `count` elements of the complex device tensor `out` to DIR/<name>.npy as [re, im] pairs of its real
    dtype (float64 for double, float32 for float): all of them when they fit this rank's share of DUMP_BYTES, else a fixed
    sample at positions (k * 2654435761 + 97) mod count, k = 0, 1, ..., in increasing order -- the same on every run."""
    import numpy as np
    import torch
    k = DUMP_BYTES // (ranks * out.element_size())
    vals = out[:count]
    if count > k:
        pos = torch.sort((torch.arange(k, dtype=torch.int64, device=out.device) * 2654435761 + 97) % count).values
        vals = vals.index_select(0, pos)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), torch.view_as_real(vals).cpu().numpy())


def flops(n0, n1, n2):
    n3 = float(n0) * n1 * n2
    return 5.0 * n3 * math.log2(n3)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference path)
# ----------------------------------------------------------------------------------------------
def cpu_forward_rate(n, budget_s=20.0, steps=None, warmup=0):
    """Times the oracle's slab pipeline on the host cores.  Full n^3 transforms when one fits the
    budget, otherwise the share of device 0 of an 8-way slab decomposition (1/8 of the work: 64
    planes of 2-D FFT + pack + its 64 y-rows of X lines) scaled by 8.  Returns a dict."""
    import numpy as np
    from oracle import FORWARD, COracle, SlabGeometry

    co = COracle()
    threads = co.num_threads()
    g = SlabGeometry(n, n, n, 1)
    a = np.zeros(n ** 3, dtype=np.complex128)
    co.fill_minstd(a[: min(a.size, 1 << 22)], 4242)   # U(0,1) heFFTe-style input (values do not affect FFT time)
    a[1 << 22:] = 0.5
    b1 = [a]
    b2 = [np.zeros_like(a)]
    t = time.perf_counter(); co.slab_execute(g, b1, b2, FORWARD); first = time.perf_counter() - t
    if steps:   # reference arm: K timed + W warm-up steps must end within a few minutes
        full = first * (steps + warmup) <= 150.0
    else:       # cpu_baseline leg: about budget_s of CPU work
        full = first <= budget_s / 2
    times = []
    if full:
        reps = steps if steps else max(1, min(5, int(budget_s / max(first, 1e-3))))
        for _ in range(warmup):
            co.slab_execute(g, b1, b2, FORWARD)
        for _ in range(reps):
            t = time.perf_counter(); co.slab_execute(g, b1, b2, FORWARD); times.append(time.perf_counter() - t)
        sample = f"{reps} full {n}^3 forward transforms (t0 2-D FFT per plane, t1 pack, t2 self copy, t3 transpose + X FFT)"
        scale = 1.0
    else:
        P = 8
        g8 = SlabGeometry(n, n, n, P)
        # only device 0's buffers take part: stage functions are called through slab_execute on a
        # 1-device geometry of the slab shape (n/8 planes for t0/t1; n/8 y-rows for t3)
        xs = n // P
        slab = SlabGeometry(xs, n, n, 1)
        reps = steps if steps else max(1, min(20, int(budget_s / max(first / P, 1e-3))))
        c1 = [a[: xs * n * n]]; c2 = [b2[0][: xs * n * n]]
        lib = co.lib
        for it in range(warmup + reps):
            t = time.perf_counter()
            lib.oracle_stage_fftZY(c1[0].ctypes.data, xs, n, n, FORWARD)
            lib.oracle_stage_pack(c1[0].ctypes.data, c2[0].ctypes.data, xs, n, n, 1, FORWARD)
            lib.oracle_stage_fftX(c2[0].ctypes.data, c1[0].ctypes.data, n, xs, n, FORWARD)
            if it >= warmup:
                times.append((time.perf_counter() - t) * P)
        sample = (f"{reps} x the share of 1 of {P} slab devices of the {n}^3 forward transform "
                  f"({xs} planes of t0/t1 + {xs}x{n} X lines of t3), time scaled by {P}")
        scale = float(P)
        del g8, slab
    best = min(times)
    mean = sum(times) / len(times)
    return {"best_s": best, "mean_s": mean, "threads": threads, "sample": sample, "scale": scale, "times": times}


def ref_forward_rate(n, steps, warmup, budget_s, precision="double"):
    """Times forward transforms of the n^3 cube by the reference tree's heFFTe (stock backend) over one slab rank per
    physical core (oracle/_ref).  `steps` timed transforms when they fit `budget_s`, fewer otherwise (said in `sample`).
    Returns None when oracle/_ref/libheffte_ref.so is absent."""
    from oracle import HeffteRef, build_ref, physical_core_cpus
    if build_ref() is None:
        return None
    ref = HeffteRef()
    cpus = physical_core_cpus(CPUS_ALLOWED)
    P = max(1, min(len(cpus), n))
    ref.pin_ranks(cpus)
    prec = 0 if precision == "double" else 1
    probe, _ = ref.time_forward(n, n, n, P, reps=1, warmup=0, algorithm="p2p_plined", precision=prec)
    per = 2.0 * probe[0] + 1e-4                        # every timed forward is followed by an untimed backward
    reps = max(1, min(steps, int(budget_s / per) - warmup))
    wu = max(0, min(warmup, int(budget_s / per) - reps))
    times, pair = ref.time_forward(n, n, n, P, reps=reps, warmup=wu, algorithm="p2p_plined", precision=prec, pair_reps=min(2, reps))
    sample = (f"{reps} full {n}^3 forward transforms by heFFTe {ref.version()} stock backend (AVX2), slab decomposition over {P} ranks "
              f"(threads behind oracle/ref_heffte/mpi.h, pinned one per physical core), reshape p2p_plined"
              + ("" if reps == steps else f"; {steps} steps requested, bounded to {reps} by the {budget_s:.0f} s budget")
              + f"; speed3d protocol (mean of forward+backward)/2 = {pair * 1e3:.1f} ms")
    return {"best_s": min(times), "mean_s": sum(times) / len(times), "threads": P, "sample": sample, "times": times, "kind": "reference",
            "logical_cpus": os.cpu_count()}


def scipy_forward_rate(n, workers, reps=3):
    """BASELINE.md section 3: scipy.fft.fftn (pocketfft, complex128) with all cores, best of `reps` warm runs."""
    import numpy as np
    import scipy.fft
    rng = np.random.default_rng(4242)
    a = rng.random((n, n, n)) + 0j
    try:   # pocketfft's worker threads inherit the caller's mask: undo an OpenMP runtime's binding of the main thread
        os.sched_setaffinity(0, CPUS_ALLOWED)
    except (AttributeError, OSError):
        pass
    scipy.fft.fftn(a, workers=workers)
    best = 1e30
    for _ in range(reps):
        t = time.perf_counter(); scipy.fft.fftn(a, workers=workers); best = min(best, time.perf_counter() - t)
    return best


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pin_openmp_threads()
    n = args.size
    r = ref_forward_rate(n, args.steps, args.warmup, budget_s=150.0, precision=args.precision)
    arm = "the reference tree's own CPU FFT: heFFTe 2.1.0 stock backend (oracle/_ref, built from /root/reference/heffte/heffteBenchmark)"
    if r is None:
        r = cpu_forward_rate(n, budget_s=20.0, steps=args.steps, warmup=args.warmup)
        r["kind"] = "port"
        arm = "CPU oracle port of the reference path (oracle/oracle_fft.c, OpenMP): oracle/_ref/libheffte_ref.so is missing"
    ms = r["mean_s"] * 1e3
    val = flops(n, n, n) * 1e-9 / r["mean_s"]
    line = {
        "impl": "reference", "metric": "3D C2C forward FFT GFlops/s (5*N^3*log2(N^3)/t)", "value": val, "unit": "GFlops/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64" if args.precision == "double" else "f32", "data": "synthetic",
        "config": {"workload": f"{n}x{n}x{n} C2C {args.precision} forward, slab decomposition over {args.gpus} GPU(s)",
                   "arm": arm, "host_threads": r["threads"], "exchange": "in-process (ranks are threads)", "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "GFlops/s", "cores": r["threads"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": val, "unit": "GFlops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_dfft_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import distributedfft_b200 as dfft

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torchrun --nproc-per-node N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the dfft arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    boot = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        boot = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.size
    prec = dfft.DOUBLE if args.precision == "double" else dfft.FLOAT
    tdt = torch.complex128 if prec == dfft.DOUBLE else torch.complex64
    esz = 16 if prec == dfft.DOUBLE else 8
    P = world
    tot, _, counts = dfft.fft_mpi_init([n, n, n], P)
    if tot != P:
        raise SystemExit(f"{n}^3 cannot use {P} devices (library suggests {tot})")
    maxc = dfft.getMaxDataCount(n, n, n, P, rank == P - 1)

    comm = None
    if P > 1:
        def allgather(b):
            out = [None] * world
            dist.all_gather_object(out, b, group=boot)
            return out
        comm = dfft.BootstrapComm(rank, P, allgather)

    # synthetic input: U(0,1) real/imag, seeded per rank; inputs (2 GiB at 512^3) are larger than L2 (126 MB)
    gen = torch.Generator(device=dev); gen.manual_seed(4242 + rank)
    tin = torch.empty(maxc, dtype=tdt, device=dev)
    torch.view_as_real(tin).uniform_(0.0, 1.0, generator=gen)
    tout = torch.empty(maxc, dtype=tdt, device=dev)
    torch.cuda.synchronize(dev)
    flags = {"auto": dfft.EXCHANGE_AUTO, "p2p": dfft.EXCHANGE_P2P, "nccl": dfft.EXCHANGE_NCCL}[args.exchange]
    if args.no_fuse:
        flags |= dfft.NO_FUSE
    if args.fuse:
        flags |= dfft.FORCE_FUSE
    if args.overlap:
        flags |= dfft.OVERLAP_X
    if args.no_pipeline:
        flags |= dfft.NO_PIPELINE
    # watchdog: a host-side hang in plan creation or the first executes (round 1's failure) ends the process with a traceback after
    # 10 minutes instead of holding the box until the driver's limit; device-side waits have their own 120 s bound (SpinGuard)
    import faulthandler
    faulthandler.dump_traceback_later(600, exit=True)
    plan = dfft.fft_mpi_plan_dft_c2c_3d(n, n, n, tin.data_ptr(), tout.data_ptr(), comm, rank, P, dfft.FORWARD, prec, flags)
    stream = torch.cuda.ExternalStream(plan.stream, device=dev)

    for _ in range(max(args.warmup, 3)):
        plan.execute()
    plan.synchronize()
    faulthandler.cancel_dump_traceback_later()

    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        plan.execute()
    e1.record(stream)
    plan.synchronize()
    barrier()
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs:   # the last timed step's result: this rank's y-slab of the spectrum, [y_l][z][x]
        dump_output(args.dump_outputs, f"spectrum_rank{rank}", tout, plan.out_count, P)
    ms_per_step = total_ms / args.steps
    stage = [max_over_ranks(x) for x in plan.timings()]
    passes = [max_over_ranks(x) for x in plan.pass_timings()]
    launches = plan.launches * args.steps

    # per-pass averages over a few more executes (events bracket each launch on the plan's stream)
    acc = [0.0, 0.0, 0.0]
    reps = 5
    for _ in range(reps):
        plan.execute()
        pt = plan.pass_timings()
        acc = [a + b for a, b in zip(acc, pt)]
    passes_avg = [max_over_ranks(a / reps) for a in acc]

    e2e = None
    plan2 = None
    hbuf = []
    if not args.no_e2e:
        # e2e: pinned HOST buffers through the C ABI; every step does its own H2D + transform + D2H inside the timed
        # region.  Two plans (two device buffer sets, two pinned buffer pairs) are driven alternately with
        # dfft_execute_host_async so that step i's D2H overlaps step i+1's H2D (PCIe is full duplex); "serial" is the
        # same loop through the synchronous dfft_execute_host of one plan.
        in_count, out_count = plan.in_count, plan.out_count
        tin2 = torch.empty(maxc, dtype=tdt, device=dev)
        tin2.copy_(tin)
        torch.cuda.synchronize(dev)
        plan2 = dfft.fft_mpi_plan_dft_c2c_3d(n, n, n, tin2.data_ptr(), None, comm, rank, P, dfft.FORWARD, prec, flags)   # in place
        hbuf = [(dfft.fft_mpi_alloc_local_memory(in_count, dfft.ALLOC_CPU, prec), dfft.fft_mpi_alloc_local_memory(out_count, dfft.ALLOC_CPU, prec))
                for _ in range(2)]
        for h_in, _ in hbuf:
            dfft.memcpy_dtoh(h_in, tin.data_ptr(), in_count * esz)
        plans = [plan, plan2]
        e2e_steps = 2 * max(2, min(args.steps, 16) // 2)
        for k in range(2):
            plans[k].execute_host(*hbuf[k])   # warm-up (first touch of the pinned pages)
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(2, e2e_steps // 4)):
            plan.execute_host(*hbuf[0])
        barrier()
        e2e_serial_s = max_over_ranks((time.perf_counter() - t0) / max(2, e2e_steps // 4))
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            plans[k % 2].execute_host_async(*hbuf[k % 2])
        plan.synchronize(); plan2.synchronize()
        barrier()
        e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    sampler.stop()
    clocks = sampler.summary()

    F = flops(n, n, n)
    if not args.no_e2e:
        e2e = {"value": F * 1e-9 / e2e_s, "unit": "GFlops/s", "ms_per_step": e2e_s * 1e3,
               "h2d_bytes_per_step": int(in_count * esz), "d2h_bytes_per_step": int(out_count * esz), "steps": e2e_steps,
               "mode": "2 plans in flight (dfft_execute_host_async): step i D2H overlaps step i+1 H2D",
               "serial_ms_per_step": e2e_serial_s * 1e3, "serial_value": F * 1e-9 / e2e_serial_s}
    value = F * 1e-9 / (ms_per_step * 1e-3)
    M = float(n) ** 3 / P
    peak, peak_src = measured_peak()
    slab_bytes = 2.0 * esz * M                      # one read + one write of the local slab (SURVEY 8d: per axis pass)
    if plan.pipeline_parts:
        # the forward transform of a device is a two-stream pipeline of part kernels (send side: Z, Y parts with the pack and the
        # peer stores / ncclAlltoAll; receive side: X parts): no single kernel dominates, the roofline is quoted on the whole
        # transform with SURVEY 8(d)'s algorithmic bytes (6 + 2) * E * M per GPU
        kernels = [(("whole forward transform, chain of two-role kernels over %d z-parts ([Z + Y0] [Y1 + X0] ... [X last]; fft_fused2_kernel, fft_fused_yx_kernel)" if plan.pipeline_chain else
                     "whole forward transform, stream-pipelined over %d z-parts (send side: Z + Y/pack/exchange parts; receive side: X parts)") % plan.pipeline_parts,
                    ms_per_step, 4 * slab_bytes, 4 * slab_bytes, "fwd_pipelined")]
    elif P > 1 and not plan.overlapped:
        # multi-GPU, plain schedule: t0 (Z + Y + NVLink peer stores in one kernel) is NVLink-bound, not HBM-bound, so a per-kernel
        # HBM fraction would mislead; SURVEY 8(d) defines the multi-GPU roofline on the whole transform: (6 + 2) * E * M / t_forward
        kernels = [("whole forward transform (fused Z+Y with NVLink peer stores, gate, X pass); t0 %.3f ms, X %.3f ms" % (passes_avg[0], passes_avg[2]),
                    ms_per_step, 4 * slab_bytes, 4 * slab_bytes, "fwd_multi")]
    elif plan.overlapped:
        # the whole forward transform of a device is ONE kernel (Z, Y with peer stores, X behind arrival flags): compulsory
        # HBM traffic = slab read + intermediate write-back + receive-buffer read + result write = 4*E*M
        kernels = [("whole forward transform (fft_fused3_kernel: Z + Y/peer-store + X roles)", passes_avg[0], 2 * slab_bytes, 3 * slab_bytes, "fwd_overlapped")]
    elif plan.fused:
        # t0 is ONE kernel doing the Z and Y passes with the intermediate resident in L2: its compulsory HBM
        # traffic is one read + one write of the slab (2*E*M); by SURVEY 8d's per-pass convention it does 4*E*M.
        kernels = [("t0 fused Z+Y (fft_fused2_kernel: contiguous + strided role, intermediate L2-resident)", passes_avg[0], slab_bytes, 2 * slab_bytes, "t0_fused"),
                   ("X pass (strided load + transposed store, fft_tile_kernel MAP_C->MAP_T)", passes_avg[2], slab_bytes, slab_bytes, "x")]
    else:
        tm = plan.tma_mask
        kn = lambda bit, tma, reg: tma if tm & bit else reg
        kernels = [(kn(1, "Z pass (contiguous lines, fft_tma_pass_kernel TMA_Z: TMA ring)", "Z pass (contiguous, fft_tile_kernel MAP_T)"), passes_avg[0], slab_bytes, slab_bytes, kn(1, "z_tma", "z")),
                   (kn(2, "Y pass (strided columns, fft_tma_pass_kernel TMA_Y: 3-D tensor TMA ring, in place)", "Y pass (strided + fused pack, fft_tile_kernel MAP_C)"), passes_avg[1], slab_bytes, slab_bytes, kn(2, "y_tma", "y")),
                   (kn(4, "X pass (strided load + transposed store, fft_tma_pass_kernel TMA_XF)", "X pass (strided load + transposed store, fft_tile_kernel MAP_C->MAP_T)"), passes_avg[2], slab_bytes, slab_bytes, kn(4, "x_tma", "x"))]
    kname, kms, alg_bytes, conv_bytes, kkey = max(kernels, key=lambda k: k[1])
    achieved = alg_bytes / (kms * 1e-3) * 1e-9
    traffic = None
    try:   # ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, captured under profiles/ (see profiles/traffic.json)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(f"{n}^3:{args.precision}:P{P}:{kkey}")
    except Exception:
        pass
    transform_bytes = (6.0 + (2.0 if P > 1 else 0.0)) * esz * M   # SURVEY 8(d) / BASELINE.md: (6 + 2*[P>1]) * E * M per GPU
    line = {
        "metric": "3D C2C forward FFT GFlops/s (5*N^3*log2(N^3)/t)", "value": value, "unit": "GFlops/s",
        "n_gpus": P, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64" if prec == dfft.DOUBLE else "f32", "data": "synthetic",
        "config": {"workload": f"{n}x{n}x{n} C2C {args.precision} forward, slab decomposition over {P} GPU(s)",
                   "exchange": {1: "p2p-fused", 2: "nccl", 3: "staged"}[plan.exchange] if P > 1 else "none",
                   "l2": "inputs (%.2f GiB per GPU) exceed the 126 MB L2; no flush needed" % (M * esz / 2 ** 30),
                   "parallelism": f"slab{P}", "pipeline_parts": plan.pipeline_parts,
                   "pipeline": ("kernel-chain" if plan.pipeline_chain else "two-stream") if plan.pipeline_parts else "none", "t0": "overlapped-single-kernel" if plan.overlapped else ("fused-L2" if plan.fused else "two-sweep")},
        "stage_ms": {"t0": stage[0], "t1": stage[1], "t2": stage[2], "t3": stage[3], "total": stage[4]},
        "pass_ms": ({"send_side_z_y_parts": passes_avg[0], "receive_side_x_parts_span": passes_avg[2]} if plan.pipeline_parts else
                    {"forward_single_kernel": passes_avg[0]} if plan.overlapped else {"t0_fused_zy": passes_avg[0], "x": passes_avg[2]} if plan.fused else
                    {"z": passes_avg[0], "y": passes_avg[1], "x": passes_avg[2]}),
        "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                     "per_pass_convention_bytes_per_launch": conv_bytes, "kernel_ms": kms,
                     "peak_source": peak_src,
                     "transform": {"achieved": transform_bytes / (ms_per_step * 1e-3) * 1e-9,
                                   "frac": transform_bytes / (ms_per_step * 1e-3) * 1e-9 / peak,
                                   "algorithmic_bytes": transform_bytes}},
        "e2e": e2e,
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if P == 1 and rank == 0 and not args.no_cpu:
        # reported baseline (not the target): the reference tree's heFFTe on the host cores, bounded to ~20 s; beside it the
        # OpenMP oracle port and scipy's pocketfft (BASELINE.md section 3), a few seconds each
        pin_openmp_threads()   # affects the oracle port's OpenMP runtime, which starts below; torch's runtime is already up
        r = ref_forward_rate(n, steps=5, warmup=1, budget_s=20.0, precision=args.precision)
        kind = "reference"
        if r is None:
            r = cpu_forward_rate(n, budget_s=15.0)
            kind = "port"
        line["cpu_baseline"] = {"value": F * 1e-9 / r["best_s"], "unit": "GFlops/s", "cores": r["threads"], "kind": kind, "sample": r["sample"]}
        others = {}
        try:
            if kind == "reference":
                rp = cpu_forward_rate(n, budget_s=6.0)
                others["oracle_port_openmp"] = {"value": F * 1e-9 / rp["best_s"], "threads": rp["threads"], "sample": rp["sample"]}
            from oracle import physical_core_cpus
            w = len(physical_core_cpus(CPUS_ALLOWED))
            others["scipy_fft_fftn"] = {"value": F * 1e-9 / scipy_forward_rate(n, w, reps=2), "workers": w, "sample": f"scipy.fft.fftn complex128 {n}^3, best of 2 warm runs"}
        except Exception as exc:   # the extra legs never take the bench line down
            others["error"] = repr(exc)
        line["cpu_baseline"]["other_cpu_ffts"] = others
    if rank == 0:
        print(json.dumps(line))
    for h_in, h_out in hbuf:
        dfft.lib().dfft_free_local(h_in, dfft.ALLOC_CPU)
        dfft.lib().dfft_free_local(h_out, dfft.ALLOC_CPU)
    if plan2 is not None:
        plan2.destroy()
    plan.destroy()
    if comm is not None:
        comm.destroy()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="dfft", choices=["dfft", "reference"])
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--precision", default="double", choices=["double", "float"])
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (large sizes: 4 pinned slabs per rank)")
    ap.add_argument("--no-fuse", action="store_true", help="run t0 as two HBM sweeps (Z pass, Y pass) instead of the fused kernel")
    ap.add_argument("--overlap", action="store_true", help="EXPERIMENTAL: whole forward transform as one kernel, t3 overlapped behind per-part arrivals (P2P, N > 1)")
    ap.add_argument("--no-pipeline", action="store_true", help="P > 1: disable the stream-pipelined z-part forward path (t2/t3 then run after t0)")
    ap.add_argument("--fuse", action="store_true", help="force the fused L2-resident t0 kernel (default: only with the P2P exchange)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the spectrum the last step computed as DIR/spectrum_rank<r>.npy "
                    "([re, im] pairs; a fixed sample when the whole would exceed %d MB); the input is the same on every run" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "dfft":
        ap.error("--dump-outputs writes the outputs of the dfft arm")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_dfft_arm(args)


if __name__ == "__main__":
    sys.exit(main())
