"""Python face of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

Two independent restatements of the reference's `3dmpifft_opt` path live here:

* `COracle`   -- ctypes binding of oracle_fft.c (own Stockham engine + the reference's stage
                 index maps; multi-threaded; also the `cpu_baseline` / `--impl reference` arm).
* `NumpySlab` -- the same stage boundaries written with numpy index arithmetic and numpy's
                 pocketfft for the math.  It shares no code with oracle_fft.c, so agreement of
                 the two (tests/test_oracle.py) checks both the engine and the layout maps.

Both are PINNED on executed reference code (tests/test_oracle_ref3d.py, tests/test_oracle_ref.py):
* `Ref3dmpifft` -- the reference's own 3dmpifft_opt sources (fft_mpi_3d_api.cpp, kernel_func.cpp, the cuTranspose kernels)
                 compiled in place against a HIP-on-CPU shim (oracle/ref_3dmpifft) and run on host memory: both plan
                 buffers after every stage, the exchange tables, the count helpers;
* `HeffteRef`  -- the reference tree's heFFTe 2.1.0 (stock CPU backend, oracle/ref_heffte): whole 3-D spectra; also the CPU
                 arm of bench.py.

Layouts follow SURVEY.md Appendix A; reference citations are on each function
(paths relative to /root/reference).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from dataclasses import dataclass

import numpy as np

FORWARD = 1    # 3dmpifft_opt/include/fft_mpi_common.h:18
BACKWARD = -1  # fft_mpi_common.h:19

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle_fft.so")


def build_oracle(force: bool = False) -> str:
    """Compile oracle_fft.c with the committed Makefile (gcc is in the image)."""
    src = os.path.join(_HERE, "oracle_fft.c")
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-s", "liboracle_fft.so"], check=True)
    return _LIB


def ceil_div(a: int, b: int) -> int:
    return -(-a // b)


@dataclass
class SlabGeometry:
    """Slab bookkeeping of fft_mpi_3d_api.cpp:56-66, 89-91 for P devices."""
    n0: int
    n1: int
    n2: int
    P: int

    @property
    def xd(self): return ceil_div(self.n0, self.P)
    @property
    def yd(self): return ceil_div(self.n1, self.P)
    @property
    def last_n0(self): return self.n0 - (self.P - 1) * self.xd
    @property
    def last_n1(self): return self.n1 - (self.P - 1) * self.yd
    def n0l(self, p): return self.last_n0 if p == self.P - 1 else self.xd
    def n1l(self, q): return self.last_n1 if q == self.P - 1 else self.yd

    def max_count(self, p):
        """getMaxDataCount, fft_mpi_3d_api.cpp:289-316"""
        return max(self.n0l(p) * self.n1 * self.n2, self.n0 * self.n1l(p) * self.n2)

    def in_count(self, p):
        """getDataCountForNode, fft_mpi_3d_api.cpp:274-287"""
        return self.n0l(p) * self.n1 * self.n2

    def out_count(self, q):
        return self.n0 * self.n1l(q) * self.n2


def proper_device_num(n0: int, wanted: int) -> int:
    """getProperDeviceNum, fft_mpi_3d_api.cpp:232-272 (single rank)."""
    if n0 % wanted == 0:
        return wanted
    per = n0 // wanted + 1
    dev = n0 // per
    if n0 % per:
        dev += 1
    return dev


# ------------------------------------------------------------------------------------------
# numpy restatement (independent of oracle_fft.c)
# ------------------------------------------------------------------------------------------
class NumpySlab:
    def __init__(self, n0, n1, n2, P):
        self.g = SlabGeometry(n0, n1, n2, P)
        if self.g.last_n0 < 1 or self.g.last_n1 < 1:
            raise ValueError("empty last slab")

    # -- helpers ---------------------------------------------------------------------------
    def scatter_input(self, A):
        """global A[x][y][z] -> per-device buf1 (flat, max_count long)"""
        g = self.g
        out = []
        for p in range(g.P):
            b = np.zeros(g.max_count(p), dtype=A.dtype)
            sl = A[p * g.xd: p * g.xd + g.n0l(p)].reshape(-1)
            b[: sl.size] = sl
            out.append(b)
        return out

    def gather_forward_output(self, buf2):
        """per-device [y_l][z][x] -> global spectrum S[x][y][z]"""
        g = self.g
        S = np.empty((g.n0, g.n1, g.n2), dtype=buf2[0].dtype)
        for q in range(g.P):
            blk = buf2[q][: g.out_count(q)].reshape(g.n1l(q), g.n2, g.n0)
            S[:, q * g.yd: q * g.yd + g.n1l(q), :] = blk.transpose(2, 0, 1)
        return S

    def gather_natural(self, bufs):
        g = self.g
        return np.concatenate([bufs[p][: g.in_count(p)] for p in range(g.P)]).reshape(g.n0, g.n1, g.n2)

    # -- stages ----------------------------------------------------------------------------
    def t0(self, buf, p, direction):
        """fftZY, fft_mpi_3d_api.cpp:466-522: in-place 2-D transform of each local plane."""
        g = self.g
        v = buf[: g.in_count(p)].reshape(g.n0l(p), g.n1, g.n2)
        f = np.fft.fft2 if direction == FORWARD else (lambda a, axes: np.fft.ifft2(a, axes=axes) * (g.n1 * g.n2))
        buf[: g.in_count(p)] = f(v, axes=(1, 2)).reshape(-1)

    def pack_index(self, p):
        """kernel_func.cpp:73-86: packed position of every natural element of device p."""
        g = self.g
        xs = g.n0l(p)
        x, y, z = np.meshgrid(np.arange(xs), np.arange(g.n1), np.arange(g.n2), indexing="ij")
        q = y // g.yd
        w = np.where(q == g.P - 1, g.last_n1, g.yd)
        return (xs * g.yd * g.n2 * q + x * w * g.n2 + (y % g.yd) * g.n2 + z).reshape(-1)

    def t1(self, src, dst, p, direction):
        idx = self.pack_index(p)
        n = idx.size
        if direction == FORWARD:
            dst[idx] = src[:n]
        else:
            dst[:n] = src[idx]

    def t2(self, buf2, buf1, direction):
        """slabAlltoall, fft_mpi_3d_api.cpp:610-672 with the tables of :84-133."""
        g = self.g
        for s in range(g.P):
            for i in range(g.P):
                if direction == FORWARD:
                    cnt = g.n0l(s) * g.n1l(i) * g.n2
                    soff = i * g.n0l(s) * g.yd * g.n2
                    roff = s * g.xd * g.n1l(i) * g.n2
                else:
                    cnt = g.n0l(i) * g.n1l(s) * g.n2
                    soff = i * g.xd * g.n1l(s) * g.n2
                    roff = s * g.n0l(i) * g.yd * g.n2
                buf1[i][roff: roff + cnt] = buf2[s][soff: soff + cnt]

    def t3(self, buf1, buf2, q, direction):
        """fftX, fft_mpi_3d_api.cpp:524-573 (+ kernels_201.cpp:46-57 / kernels_120.cpp:45-57)."""
        g = self.g
        n = g.out_count(q)
        if direction == FORWARD:
            v = buf1[:n].reshape(g.n0, g.n1l(q), g.n2).transpose(1, 2, 0)
            buf2[:n] = np.fft.fft(v, axis=2).reshape(-1)
        else:
            v = np.fft.ifft(buf1[:n].reshape(g.n1l(q), g.n2, g.n0), axis=2) * g.n0
            buf1[:n] = v.reshape(-1)  # the reference transforms bufferDev1 in place (api.cpp:561)
            buf2[:n] = v.transpose(2, 0, 1).reshape(-1)

    def execute(self, buf1, buf2, direction, stop_after=3):
        """fft_mpi_execute_dft_3d_c2c, fft_mpi_3d_api.cpp:181-214."""
        g = self.g
        if direction == FORWARD:
            for p in range(g.P): self.t0(buf1[p], p, direction)
            if stop_after == 0: return
            for p in range(g.P): self.t1(buf1[p], buf2[p], p, direction)
            if stop_after == 1: return
            self.t2(buf2, buf1, direction)
            if stop_after == 2: return
            for q in range(g.P): self.t3(buf1[q], buf2[q], q, direction)
        else:
            for q in range(g.P): self.t3(buf1[q], buf2[q], q, direction)
            if stop_after == 0: return
            self.t2(buf2, buf1, direction)
            if stop_after == 1: return
            for p in range(g.P): self.t1(buf1[p], buf2[p], p, direction)
            if stop_after == 2: return
            for p in range(g.P): self.t0(buf2[p], p, direction)


# ------------------------------------------------------------------------------------------
# ctypes binding of oracle_fft.c
# ------------------------------------------------------------------------------------------
class COracle:
    def __init__(self):
        self.lib = ctypes.CDLL(build_oracle())
        L = self.lib
        i64 = ctypes.c_longlong
        vp = ctypes.c_void_p
        L.oracle_radix_schedule.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.oracle_radix_schedule.restype = ctypes.c_int
        L.oracle_fft_batch.argtypes = [vp, ctypes.c_int, i64, i64, i64, i64, i64, ctypes.c_int]
        L.oracle_fft_batch.restype = None
        L.oracle_proper_device_num.argtypes = [i64, ctypes.c_int]
        L.oracle_proper_device_num.restype = ctypes.c_int
        L.oracle_max_data_count.argtypes = [i64, i64, i64, ctypes.c_int, ctypes.c_int]
        L.oracle_max_data_count.restype = i64
        L.oracle_exchange_table.argtypes = [i64, i64, i64, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
        L.oracle_exchange_table.restype = None
        L.oracle_slab_execute.argtypes = [ctypes.c_int, i64, i64, i64, vp, vp, ctypes.c_int, ctypes.c_int]
        L.oracle_slab_execute.restype = ctypes.c_int
        L.oracle_fill_ramp.argtypes = [vp, i64, i64]
        L.oracle_fill_minstd.argtypes = [vp, i64, ctypes.POINTER(ctypes.c_ulonglong)]
        L.oracle_roundtrip_error.argtypes = [vp, vp, i64, ctypes.c_double, ctypes.POINTER(ctypes.c_double)]
        L.oracle_roundtrip_error.restype = ctypes.c_double
        L.oracle_num_threads.restype = ctypes.c_int
        L.oracle_stage_fftZY.argtypes = [vp, i64, i64, i64, ctypes.c_int]
        L.oracle_stage_pack.argtypes = [vp, vp, i64, i64, i64, ctypes.c_int, ctypes.c_int]
        L.oracle_stage_fftX.argtypes = [vp, vp, i64, i64, i64, ctypes.c_int]
        for f in (L.oracle_stage_fftZY, L.oracle_stage_pack, L.oracle_stage_fftX):
            f.restype = None

    def radix_schedule(self, n):
        r = (ctypes.c_int * 32)()
        k = self.lib.oracle_radix_schedule(n, r)
        return list(r[:k])

    def num_threads(self):
        return int(self.lib.oracle_num_threads())

    def fft_axis(self, a: np.ndarray, axis: int, sign: int) -> np.ndarray:
        """1-D transforms along `axis` of a C-contiguous complex128 array (copy returned)."""
        a = np.ascontiguousarray(a, dtype=np.complex128).copy()
        n = a.shape[axis]
        stride = int(np.prod(a.shape[axis + 1:], dtype=np.int64))
        outer = int(np.prod(a.shape[:axis], dtype=np.int64))
        self.lib.oracle_fft_batch(a.ctypes.data, n, stride, outer * stride, stride, 1, n * stride, sign)
        return a

    def exchange_table(self, n0, n1, n2, P, dev, direction):
        arrs = [np.zeros(P, dtype=np.int64) for _ in range(4)]
        self.lib.oracle_exchange_table(n0, n1, n2, P, dev, direction, *[a.ctypes.data for a in arrs])
        return dict(zip(("scount", "soffset", "rcount", "roffset"), arrs))

    def slab_execute(self, geom: SlabGeometry, buf1, buf2, direction, stop_after=3):
        P = geom.P
        p1 = (ctypes.c_void_p * P)(*[b.ctypes.data for b in buf1])
        p2 = (ctypes.c_void_p * P)(*[b.ctypes.data for b in buf2])
        rc = self.lib.oracle_slab_execute(P, geom.n0, geom.n1, geom.n2, p1, p2, direction, stop_after)
        if rc != 0:
            raise ValueError("oracle_slab_execute failed (empty last slab?)")

    def fill_ramp(self, dst: np.ndarray, start: int):
        self.lib.oracle_fill_ramp(dst.ctypes.data, start, dst.size)

    def fill_minstd(self, dst: np.ndarray, state: int = 4242) -> int:
        st = ctypes.c_ulonglong(state)
        self.lib.oracle_fill_minstd(dst.ctypes.data, dst.size, ctypes.byref(st))
        return int(st.value)

    def roundtrip_error(self, a: np.ndarray, b: np.ndarray, n3: float):
        ab = ctypes.c_double(0)
        drv = self.lib.oracle_roundtrip_error(a.ctypes.data, b.ctypes.data, a.size, float(n3), ctypes.byref(ab))
        return float(drv), float(ab.value)


def sampled(a, k: int) -> np.ndarray:
    """k entries of the flattened `a` at fixed positions spread over it (all of it when k >= a.size).  The positions depend
    only on (a.size, k) and not on numpy's random streams, so a stored sample of a large reference output can be compared
    with the same positions of a recomputation."""
    a = np.asarray(a).reshape(-1)
    if k >= a.size:
        return a.copy()
    return a[np.unique((np.arange(k, dtype=np.int64) * 2654435761 + 97) % a.size)]   # distinct: the multiplier is a prime > a.size


def minstd_uniform(count: int, state: int = 4242):
    """numpy restatement of heffte/heffteBenchmark/test/test_fft3d.h:19-27 input
    (std::minstd_rand(4242) -> uniform_real_distribution<double>(0,1)); returns (values, state)."""
    a, m = 48271, 2147483647
    R = float(m - 1)
    out = np.empty(count, dtype=np.float64)
    s = state
    for j in range(count):
        s = (s * a) % m; lo = s - 1
        s = (s * a) % m; hi = s - 1
        out[j] = (lo + hi * R) / (R * R)
    return out, s


# ------------------------------------------------------------------------------------------
# oracle/_ref: the reference tree's own heFFTe 2.1.0 (stock CPU backend), compiled from the sources under
# /root/reference by oracle/ref_heffte/Makefile -- the EXECUTED reference that pins the restatements above
# and the `--impl reference` CPU arm of bench.py.  The .so is git-ignored and travels to the GPU box prebuilt.
# ------------------------------------------------------------------------------------------
_REF_DIR = os.path.join(_HERE, "_ref")
_REF_LIB = os.path.join(_REF_DIR, "libheffte_ref.so")
_REF_SRC = "/root/reference/heffte/heffteBenchmark"


def build_ref(force: bool = False):
    """Build oracle/_ref/libheffte_ref.so when the reference tree is present (this container); on the GPU box the
    prebuilt file is used as is.  Returns its path, or None when it neither exists nor can be built."""
    rdir = os.path.join(_HERE, "ref_heffte")
    if os.path.isdir(_REF_SRC):
        deps = [os.path.join(rdir, f) for f in ("heffte_ref.cpp", "tmpi.cpp", "mpi.h", "heffte_config.h", "Makefile")]
        if force or not os.path.exists(_REF_LIB) or os.path.getmtime(_REF_LIB) < max(os.path.getmtime(d) for d in deps):
            subprocess.run(["make", "-C", rdir, "-s", f"REF={_REF_SRC}"], check=True)
    return _REF_LIB if os.path.exists(_REF_LIB) else None


class HeffteRef:
    """ctypes binding of oracle/_ref/libheffte_ref.so (oracle/ref_heffte/heffte_ref.cpp): world-array transforms by the
    reference tree's heFFTe over P slab ranks (threads behind the mpi.h stand-in)."""
    ALGORITHMS = {"alltoallv": 0, "alltoall": 1, "p2p_plined": 2, "p2p": 3}

    def __init__(self):
        path = build_ref()
        if path is None:
            raise FileNotFoundError("oracle/_ref/libheffte_ref.so is missing and /root/reference is not available to build it")
        self.lib = ctypes.CDLL(path)
        vp, i = ctypes.c_void_p, ctypes.c_int
        self.lib.heffte_ref_fft3d_c2c.argtypes = [i, i, i, i, vp, vp, i, i, i, i]
        self.lib.heffte_ref_time.argtypes = [i, i, i, i, i, i, i, i, i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]

    def version(self):
        return int(self.lib.heffte_ref_version())

    def pin_ranks(self, cpus):
        """pin rank i to cpus[i % len(cpus)] (one CPU per physical core, see physical_core_cpus()); [] clears it"""
        arr = (ctypes.c_int * max(1, len(cpus)))(*cpus)
        self.lib.tmpi_set_cpus(arr, len(cpus))

    def fft3d(self, A: np.ndarray, P: int, direction: int = FORWARD, algorithm: str = "p2p_plined", scale_full: bool = False) -> np.ndarray:
        """A[x][y][z] (complex128 / complex64) -> its forward (direction +1) or backward spectrum, natural order"""
        prec = 0 if A.dtype == np.complex128 else 1
        A = np.ascontiguousarray(A)
        out = np.zeros_like(A)
        n0, n1, n2 = A.shape
        rc = self.lib.heffte_ref_fft3d_c2c(n0, n1, n2, P, A.ctypes.data, out.ctypes.data, direction, self.ALGORITHMS[algorithm], prec, int(scale_full))
        if rc != 0:
            raise ValueError(f"heffte_ref_fft3d_c2c failed ({rc})")
        return out

    def time_forward(self, n0, n1, n2, P, reps=3, warmup=1, algorithm="p2p_plined", precision=0, pair_reps=0):
        """returns (forward seconds per repetition, speed3d-protocol seconds = mean of (forward + backward) / 2)"""
        t = (ctypes.c_double * reps)()
        pair = ctypes.c_double(0)
        rc = self.lib.heffte_ref_time(n0, n1, n2, P, reps, warmup, pair_reps, self.ALGORITHMS[algorithm], precision, t, ctypes.byref(pair))
        if rc != 0:
            raise ValueError(f"heffte_ref_time failed ({rc})")
        return list(t), float(pair.value)


def physical_core_cpus(allowed=None):
    """One logical CPU per physical core among `allowed` (default: the CPUs the calling thread may run on -- pass the
    process's set captured at start-up when an OpenMP runtime may have bound the main thread since); hyperthread
    siblings are dropped."""
    if allowed is None:
        try:
            allowed = sorted(os.sched_getaffinity(0))
        except AttributeError:
            allowed = list(range(os.cpu_count() or 1))
    seen, out = set(), []
    for c in allowed:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                key = f.read().strip()
        except OSError:
            key = str(c)
        if key not in seen:
            seen.add(key)
            out.append(c)
    return out


# ------------------------------------------------------------------------------------------
# oracle/_ref/libref3dmpifft.so (+ libtemplatefft_cpu.so, libhipcpu.so): the reference's OWN HOT-PATH SOURCES executed on the
# CPU.  oracle/ref_3dmpifft/Makefile compiles 3dmpifft_opt/include/fft_mpi_3d_api.cpp, kernel_func.cpp,
# fast_transpose/kernels_{201,120}.cpp and the FFT engine templateFFT/src/templateFFT.cpp where they lie under /root/reference
# against a HIP-on-CPU shim (kernel launches run on fibers, so __shared__ / __syncthreads work; the kernels the engine generates
# at run time are compiled with g++ in place of hiprtc).  Plan creation, exchange tables, fftZY, the FFT kernels,
# localTransposeUneven + pack kernels, slabAlltoall, fftX + cuTranspose kernels are the reference's code.
# ------------------------------------------------------------------------------------------
_REF3D_LIB = os.path.join(_REF_DIR, "libref3dmpifft.so")
_REF3D_SRC = "/root/reference/3dmpifft_opt/include"


def build_ref3d(force: bool = False):
    """Build oracle/_ref/libref3dmpifft.so when the reference tree is present; else use the prebuilt file.  Returns its
    path, or None when it neither exists nor can be built."""
    rdir = os.path.join(_HERE, "ref_3dmpifft")
    if os.path.isdir(_REF3D_SRC):
        deps = [os.path.join(rdir, f) for f in ("ref3d_glue.cpp", "hipcpu.cpp", "tfft_engine.cpp", "Makefile", "mpi.h", "rocfft.h", "hipfft.h", "rccl.h",
                                                "hip/hip_runtime.h", "hip/hiprtc.h")]
        libs = [_REF3D_LIB, os.path.join(_REF_DIR, "libhipcpu.so"), os.path.join(_REF_DIR, "libtemplatefft_cpu.so"), os.path.join(_REF_DIR, "distFFT_ref")]
        if force or not all(os.path.exists(l) for l in libs) or min(os.path.getmtime(l) for l in libs) < max(os.path.getmtime(d) for d in deps):
            subprocess.run(["make", "-C", rdir, "-s", "REF=/root/reference"], check=True)
    return _REF3D_LIB if os.path.exists(_REF3D_LIB) else None


class Ref3dmpifft:
    """ctypes binding of oracle/_ref/libref3dmpifft.so (oracle/ref_3dmpifft/ref3d_glue.cpp).  Sizes are test-sized: every GPU
    thread of every kernel launch is a fiber and the FFT arithmetic is an O(N^2) DFT."""

    def __init__(self):
        path = build_ref3d()
        if path is None:
            raise FileNotFoundError("oracle/_ref/libref3dmpifft.so is missing and /root/reference is not available to build it")
        self.lib = ctypes.CDLL(path)
        i, vp = ctypes.c_int, ctypes.c_void_p
        self.lib.ref3d_run.argtypes = [i, i, i, i, i, vp, vp, vp, vp]
        self.lib.ref3d_max_data_count.restype = ctypes.c_longlong
        self.lib.ref3d_max_data_count.argtypes = [i, i, i, i, i]
        self.lib.ref3d_proper_device_num.argtypes = [ctypes.c_longlong, i, i]
        self.lib.ref3d_set_engine.argtypes = [i]
        self.lib.ref3d_engine_fft.argtypes = [i, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong, i, vp]
        self.engine = self.set_engine("templatefft")

    def set_engine(self, name: str) -> str:
        """'templatefft': the reference's own FFT engine (templateFFT/src/templateFFT.cpp: its generator and the kernels it emits,
        compiled with g++ at run time; needs g++); 'dft': a plain DFT behind the same entry points.  Returns the engine in effect
        ('dft' when libtemplatefft_cpu.so is absent)."""
        got = self.lib.ref3d_set_engine(1 if name == "templatefft" else 0)
        self.engine = "templatefft" if got == 1 else "dft"
        return self.engine

    def engine_schedule(self, n):
        """(radices, uploads) the reference's generator chose for n points (templateFFT.cpp FFTScheduler), or None when it does
        not take the length"""
        r = (ctypes.c_int * 64)()
        up = ctypes.c_int(0)
        k = self.lib.ref3d_engine_schedule(ctypes.c_longlong(n), r, 64, ctypes.byref(up))
        return None if k < 0 else (list(r[:k]), int(up.value))

    def engine_used(self, n0, n1, n2) -> str:
        """which FFT arithmetic execute() runs for this size"""
        def smooth7(n):
            for p in (2, 3, 5, 7):
                while n % p == 0:
                    n //= p
            return n == 1
        return self.engine if self.engine == "dft" or all(smooth7(n) for n in (n0, n1, n2)) else "dft"

    def engine_fft(self, a: np.ndarray, fftdim: int = 1, inverse: bool = False):
        """The reference's FFT engine alone (the templateFFT batch-test surface): transform over the last `fftdim` axes of the
        C-ordered complex128 array `a`, leading axes are batches.  Returns the result, or None when the generator does not
        take the size (a prime factor > 7)."""
        x = np.ascontiguousarray(a, dtype=np.complex128).copy()
        shp = x.shape
        s0 = shp[-1]
        s1 = shp[-2] if x.ndim >= 2 else 1
        s2 = int(np.prod(shp[:-2])) if x.ndim > 2 else 1
        rc = self.lib.ref3d_engine_fft(fftdim, s0, s1, s2, int(inverse), x.ctypes.data)
        if rc == -3:
            return None
        if rc != 0:
            raise RuntimeError(f"ref3d_engine_fft failed ({rc})")
        return x

    def max_data_count(self, n0, n1, n2, P, is_last):
        """getMaxDataCount, fft_mpi_3d_api.cpp:289-316, as compiled from the reference"""
        return int(self.lib.ref3d_max_data_count(n0, n1, n2, P, int(is_last)))

    def proper_device_num(self, n0, wanted, have=64):
        """getProperDeviceNum, fft_mpi_3d_api.cpp:232-272 (one rank, `have` devices present)"""
        return int(self.lib.ref3d_proper_device_num(n0, wanted, have))

    def tables(self, n0, n1, n2, P, direction):
        """TransInfo of every device as filled by the reference's plan creation (fft_mpi_3d_api.cpp:84-133), no transform:
        tables[p][q] = (scount, soffset, rcount, roffset)"""
        t = np.zeros((P, P, 4), dtype=np.int64)
        if self.lib.ref3d_tables(n0, n1, n2, P, direction, ctypes.c_void_p(t.ctypes.data)) != 0:
            raise ValueError("ref3d_tables failed")
        return t

    def execute(self, geom: SlabGeometry, inputs, direction, stages: bool = False):
        """Run the reference driver's sequence (fftSpeed3d_c2c.cpp:42-102) on P "devices".  inputs[p]: max_count(p) complex128
        (x-slabs forward, y-slabs backward).  Returns (outputs, tables, dumps): outputs[p] = the device's out buffer,
        tables[p][q] = (scount, soffset, rcount, roffset) of plan p towards q, dumps[p][stage] = (bufferDev1, bufferDev2)
        after each of the four stages in execution order when stages=True (the stage functions are then called one by one),
        else None (the reference's own fft_mpi_execute_dft_3d_c2c runs)."""
        P = geom.P
        ins = [np.ascontiguousarray(b, dtype=np.complex128) for b in inputs]
        assert all(b.size == geom.max_count(p) for p, b in enumerate(ins))
        outs = [np.zeros(geom.max_count(p), dtype=np.complex128) for p in range(P)]
        tables = np.zeros((P, P, 4), dtype=np.int64)
        arr = ctypes.c_void_p * P
        dumps = dp = None
        if stages:
            dumps = [[(np.zeros(geom.max_count(p), dtype=np.complex128), np.zeros(geom.max_count(p), dtype=np.complex128)) for _ in range(4)] for p in range(P)]
            dp = (ctypes.c_void_p * (P * 8))(*[dumps[p][s][w].ctypes.data for p in range(P) for s in range(4) for w in range(2)])
        rc = self.lib.ref3d_run(geom.n0, geom.n1, geom.n2, P, direction, arr(*[b.ctypes.data for b in ins]), arr(*[b.ctypes.data for b in outs]),
                                dp, tables.ctypes.data)
        if rc != 0:
            raise ValueError(f"ref3d_run failed ({rc}): the reference would not run {geom.n0}x{geom.n1}x{geom.n2} on {P} devices")
        return outs, tables, dumps
