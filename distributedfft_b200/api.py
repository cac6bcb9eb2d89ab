"""ctypes binding of libdfft.so mirroring the reference's slab-FFT API.

Reference surface (3dmpifft_opt/include/fft_mpi_3d_api.h:68-74, fft_mpi_common.h:15-22):
    fft_mpi_init, fft_mpi_plan_dft_c2c_3d, fft_mpi_execute_dft_3d_c2c, fft_mpi_destroy_plan,
    fft_mpi_alloc_local_memory, fft_mpi_local_size_3d, fft_mpi_cleanup, getMaxDataCount,
    FORWARD / BACKWARD, ALLOC_CPU / ALLOC_DEV.
Same names, argument meaning and error behaviour (errors raise DfftError instead of exit()).
Device memory is handled as raw pointers; callers may pass torch CUDA tensors' data_ptr().
"""
from __future__ import annotations

import ctypes
import os

FORWARD = 1
BACKWARD = -1
ALLOC_CPU = 1
ALLOC_DEV = -1
DOUBLE = 0
FLOAT = 1
EXCHANGE_AUTO, EXCHANGE_P2P, EXCHANGE_NCCL, EXCHANGE_STAGED = 0, 1, 2, 3
SCALE_BACKWARD = 4
NO_FUSE = 8
FORCE_FUSE = 16
OVERLAP_X = 32
NATURAL_SPECTRUM = 64
DRY_RUN = 128
NO_PIPELINE = 256
NO_TMA = 512
FORCE_PIPELINE = 1024

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdfft.so")

__all__ = [
    "FORWARD", "BACKWARD", "ALLOC_CPU", "ALLOC_DEV", "DOUBLE", "FLOAT", "EXCHANGE_AUTO", "EXCHANGE_P2P",
    "EXCHANGE_NCCL", "EXCHANGE_STAGED", "SCALE_BACKWARD", "NO_FUSE", "FORCE_FUSE", "OVERLAP_X", "NATURAL_SPECTRUM", "DRY_RUN", "NO_PIPELINE", "NO_TMA", "FORCE_PIPELINE", "DfftError", "lib", "LIB_PATH", "Plan", "LocalComm",
    "BootstrapComm", "fft_mpi_init", "fft_mpi_plan_dft_c2c_3d", "fft_mpi_execute_dft_3d_c2c", "fft_mpi_destroy_plan",
    "fft_mpi_alloc_local_memory", "fft_mpi_local_size_3d", "fft_mpi_cleanup", "getMaxDataCount", "supported_lengths",
    "fft_lines", "lines_ops", "LinesPlan", "length_kind", "length_schedule", "fused_kinds", "memcpy_htod", "memcpy_dtoh", "exchange_table", "comm_allgather",
]


class DfftError(RuntimeError):
    pass


_ALLGATHER = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)
_lib = None


def lib():
    """Load libdfft.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DfftError(f"{LIB_PATH} is missing: build it with `python -m distributedfft_b200.build` "
                        "(there is no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    ll, i, vp, u = ctypes.c_longlong, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint
    P = ctypes.POINTER
    L.dfft_last_error.restype = ctypes.c_char_p
    L.dfft_version.restype = i
    L.dfft_supported_lengths.argtypes = [i, P(i), i]
    L.dfft_init.argtypes = [P(ll), i, P(i), P(i), P(ll)]
    L.dfft_max_data_count.argtypes = [ll, ll, ll, i, i]
    L.dfft_max_data_count.restype = ll
    L.dfft_local_size_3d.argtypes = [ll, ll, ll, i, i, P(ll), P(ll), P(ll), P(ll)]
    L.dfft_local_size_3d.restype = ll
    L.dfft_alloc_local.argtypes = [ll, i, i]
    L.dfft_alloc_local.restype = vp
    L.dfft_free_local.argtypes = [vp, i]
    L.dfft_comm_create_local.argtypes = [i, P(vp)]
    L.dfft_comm_create_bootstrap.argtypes = [i, i, _ALLGATHER, vp, P(vp)]
    L.dfft_comm_destroy.argtypes = [vp]
    L.dfft_comm_allgather.argtypes = [vp, i, vp, vp, ctypes.c_size_t]
    L.dfft_exchange_table.argtypes = [ll, ll, ll, i, i, i, P(ll), P(ll), P(ll), P(ll)]
    L.dfft_plan_c2c_3d.argtypes = [ll, ll, ll, vp, vp, vp, i, i, i, i, u, P(vp)]
    for name in ("dfft_execute", "dfft_synchronize", "dfft_destroy", "dfft_plan_launches", "dfft_plan_exchange", "dfft_plan_fused", "dfft_plan_pipeline_parts", "dfft_plan_tma_mask", "dfft_plan_pipeline_chain"):
        getattr(L, name).argtypes = [vp]
    L.dfft_execute_stage.argtypes = [vp, i]
    L.dfft_execute_host.argtypes = [vp, vp, vp]
    L.dfft_execute_host_async.argtypes = [vp, vp, vp]
    L.dfft_get_timings.argtypes = [vp, P(ctypes.c_double)]
    L.dfft_get_pass_timings.argtypes = [vp, P(ctypes.c_double)]
    L.dfft_plan_buffers.argtypes = [vp, P(vp), P(vp)]
    L.dfft_plan_counts.argtypes = [vp, P(ll), P(ll), P(ll)]
    L.dfft_plan_stream.argtypes = [vp]
    L.dfft_plan_stream.restype = vp
    L.dfft_fft_lines.argtypes = [vp, i, ll, ll, ll, ll, ll, i, i]
    L.dfft_lines_plan_create.argtypes = [i, ll, ll, ll, ll, ll, i, P(vp)]
    L.dfft_lines_plan_create_2d.argtypes = [i, i, ll, i, P(vp)]
    L.dfft_lines_execute.argtypes = [vp, vp, i]
    L.dfft_lines_synchronize.argtypes = [vp]
    L.dfft_lines_destroy.argtypes = [vp]
    L.dfft_lines_stream.argtypes = [vp]
    L.dfft_lines_stream.restype = vp
    L.dfft_length_kind.argtypes = [i, i]
    L.dfft_debug_plan_ops.argtypes = [vp, ctypes.c_char_p, ll]
    L.dfft_debug_plan_ops.restype = ll
    L.dfft_debug_lines_ops.argtypes = [i, ll, ll, ll, ll, ll, i, i, i, ctypes.c_char_p, ll]
    L.dfft_debug_lines_ops.restype = ll
    L.dfft_length_schedule.argtypes = [i, i, P(ctypes.c_int), i]
    L.dfft_debug_fused_kinds.argtypes = [i, i]
    L.dfft_debug_fused3_order.argtypes = [ll, ll, i, i, i, i, i, ll, P(ll)]
    L.dfft_debug_fused3_order.restype = ll
    L.dfft_memcpy.argtypes = [vp, vp, ctypes.c_size_t, i]
    L.dfft_debug_timeline.argtypes = [vp, P(ctypes.c_double)]
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise DfftError(f"{what} failed ({rc}): {lib().dfft_last_error().decode()}")


def supported_lengths(precision=DOUBLE):
    n = lib().dfft_supported_lengths(precision, None, 0)
    arr = (ctypes.c_int * n)()
    lib().dfft_supported_lengths(precision, arr, n)
    return list(arr)


def length_kind(n, precision=DOUBLE):
    """2 = tuned kernel, 1 = run-time-scheduled kernel (2..13-smooth lengths), 0 = unsupported."""
    return int(lib().dfft_length_kind(n, precision))


def fused_kinds(n, precision=DOUBLE):
    """bit mask of the multi-role kernels length n has (see dfft_debug_fused_kinds); -1 if unsupported"""
    return int(lib().dfft_debug_fused_kinds(n, precision))


def length_schedule(n, precision=DOUBLE):
    """radix list the library uses for length n ([] if unsupported)"""
    arr = (ctypes.c_int * 32)()
    k = lib().dfft_length_schedule(n, precision, arr, 32)
    return list(arr[:k])


def getMaxDataCount(n0, n1, n2, totalDevCount, isLastDevice):
    """getMaxDataCount, fft_mpi_3d_api.cpp:289-316"""
    return int(lib().dfft_max_data_count(n0, n1, n2, totalDevCount, int(bool(isLastDevice))))


def fft_mpi_init(N, iniDeviceNumInNode):
    """fft_mpi_init (fft_mpi_3d_api.cpp:3-39). Returns (newDeviceCount, newDeviceCountInNode, dataCountInNode)."""
    n = (ctypes.c_longlong * 3)(*N)
    tot, loc = ctypes.c_int(0), ctypes.c_int(0)
    counts = (ctypes.c_longlong * max(1, iniDeviceNumInNode))()
    _check(lib().dfft_init(n, iniDeviceNumInNode, ctypes.byref(tot), ctypes.byref(loc), counts), "fft_mpi_init")
    return tot.value, loc.value, list(counts[: tot.value])


def fft_mpi_local_size_3d(n0, n1, n2, totalDevCount, devIdx):
    """declared fft_mpi_3d_api.h:73; returns (alloc, local_n0, local_0_start, local_n1, local_1_start)"""
    a, b, c, d = (ctypes.c_longlong(0) for _ in range(4))
    r = lib().dfft_local_size_3d(n0, n1, n2, totalDevCount, devIdx, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c), ctypes.byref(d))
    if r < 0:
        raise DfftError("fft_mpi_local_size_3d: bad arguments")
    return int(r), a.value, b.value, c.value, d.value


def fft_mpi_alloc_local_memory(count, flag, precision=DOUBLE):
    """fft_mpi_alloc_local_memory (fft_mpi_3d_api.cpp:216-230); returns a raw pointer (int)."""
    p = lib().dfft_alloc_local(count, flag, precision)
    if not p:
        raise DfftError("fft_mpi_alloc_local_memory: " + lib().dfft_last_error().decode())
    return p


def exchange_table(n0, n1, n2, totalDevCount, devIdx, direction):
    """TransInfo of one device (fft_mpi_3d_api.cpp:84-133): dict of scount/soffset/rcount/roffset lists."""
    arrs = [(ctypes.c_longlong * totalDevCount)() for _ in range(4)]
    _check(lib().dfft_exchange_table(n0, n1, n2, totalDevCount, devIdx, direction, *arrs), "dfft_exchange_table")
    return dict(zip(("scount", "soffset", "rcount", "roffset"), (list(x) for x in arrs)))


def comm_allgather(comm, rank, payload: bytes):
    """All-gather `payload` through a dfft communicator (the plan-creation bootstrap path)."""
    n = comm.nranks
    buf = ctypes.create_string_buffer(len(payload) * n)
    _check(lib().dfft_comm_allgather(comm.handle, rank, payload, buf, len(payload)), "dfft_comm_allgather")
    return [buf.raw[i * len(payload):(i + 1) * len(payload)] for i in range(n)]


def fft_mpi_cleanup():
    lib().dfft_cleanup()


class LocalComm:
    """P device-threads of one process (the reference's GPUs-per-rank mode)."""

    def __init__(self, nranks):
        h = ctypes.c_void_p()
        _check(lib().dfft_comm_create_local(nranks, ctypes.byref(h)), "dfft_comm_create_local")
        self.handle, self.nranks = h, nranks

    def destroy(self):
        if self.handle:
            lib().dfft_comm_destroy(self.handle)
            self.handle = None


class BootstrapComm:
    """One process per GPU; `allgather(bytes) -> list[bytes]` supplied by the host program
    (e.g. torch.distributed.all_gather_object).  Stands in for the reference's MPI_Comm."""

    def __init__(self, rank, nranks, allgather):
        self._py_allgather = allgather

        def _cb(ctx, send, recv, nbytes):
            try:
                mine = ctypes.string_at(send, nbytes)
                parts = self._py_allgather(mine)
                assert len(parts) == nranks and all(len(x) == nbytes for x in parts)
                ctypes.memmove(recv, b"".join(parts), nbytes * nranks)
                return 0
            except Exception as exc:  # pragma: no cover - surfaced as DFFT_ECOMM
                print("dfft bootstrap allgather failed:", exc)
                return -1

        self._cb = _ALLGATHER(_cb)
        h = ctypes.c_void_p()
        _check(lib().dfft_comm_create_bootstrap(rank, nranks, self._cb, None, ctypes.byref(h)), "dfft_comm_create_bootstrap")
        self.handle, self.nranks, self.rank = h, nranks, rank

    def destroy(self):
        if self.handle:
            lib().dfft_comm_destroy(self.handle)
            self.handle = None


class Plan:
    """fft_mpi_3d_plan (fft_mpi_3d_api.h:11-66): bufferDev1/bufferDev2, counts, timings."""

    def __init__(self, handle):
        self.handle = handle
        b1, b2 = ctypes.c_void_p(), ctypes.c_void_p()
        _check(lib().dfft_plan_buffers(handle, ctypes.byref(b1), ctypes.byref(b2)), "dfft_plan_buffers")
        self.bufferDev1, self.bufferDev2 = b1.value, b2.value
        a, b, c = (ctypes.c_longlong(0) for _ in range(3))
        _check(lib().dfft_plan_counts(handle, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)), "dfft_plan_counts")
        self.in_count, self.out_count, self.maxDataCountInDevice = a.value, b.value, c.value

    def execute(self):
        _check(lib().dfft_execute(self.handle), "fft_mpi_execute_dft_3d_c2c")

    def execute_stage(self, stage):
        _check(lib().dfft_execute_stage(self.handle, stage), "dfft_execute_stage")

    def execute_host(self, host_in_ptr, host_out_ptr):
        _check(lib().dfft_execute_host(self.handle, host_in_ptr, host_out_ptr), "dfft_execute_host")

    def execute_host_async(self, host_in_ptr, host_out_ptr):
        _check(lib().dfft_execute_host_async(self.handle, host_in_ptr, host_out_ptr), "dfft_execute_host_async")

    def synchronize(self):
        _check(lib().dfft_synchronize(self.handle), "dfft_synchronize")

    def timings(self):
        t = (ctypes.c_double * 5)()
        _check(lib().dfft_get_timings(self.handle, t), "dfft_get_timings")
        return list(t)

    def pass_timings(self):
        t = (ctypes.c_double * 3)()
        _check(lib().dfft_get_pass_timings(self.handle, t), "dfft_get_pass_timings")
        return list(t)

    @property
    def launches(self):
        return lib().dfft_plan_launches(self.handle)

    @property
    def exchange(self):
        return lib().dfft_plan_exchange(self.handle)

    @property
    def fused(self):
        return bool(lib().dfft_plan_fused(self.handle))

    def recorded_ops(self):
        """passes recorded by the last execute of a DRY_RUN plan (list of dicts)"""
        import json
        n = lib().dfft_debug_plan_ops(self.handle, None, 0)
        buf = ctypes.create_string_buffer(int(n))
        lib().dfft_debug_plan_ops(self.handle, buf, n)
        return json.loads(buf.value.decode())

    def debug_timeline(self):
        t = (ctypes.c_double * 11)()
        _check(lib().dfft_debug_timeline(self.handle, t), "dfft_debug_timeline")
        return list(t)

    @property
    def tma_mask(self):
        """bit 0 / 1 / 2: the un-chunked Z / Y / X pass runs on the TMA-pipelined kernel"""
        return lib().dfft_plan_tma_mask(self.handle)

    @property
    def pipeline_parts(self):
        """z-parts of the stream-pipelined forward path (0 = not pipelined)"""
        return lib().dfft_plan_pipeline_parts(self.handle)

    @property
    def pipeline_chain(self):
        """the z-parts run as a chain of two-role kernels on one stream (Y part k + X part k-1 per kernel)"""
        return bool(lib().dfft_plan_pipeline_chain(self.handle))

    @property
    def overlapped(self):
        """forward transform runs as the single overlapped kernel (OVERLAP_X, experimental)"""
        return lib().dfft_plan_fused(self.handle) == 2

    @property
    def stream(self):
        return lib().dfft_plan_stream(self.handle)

    def destroy(self):
        if self.handle:
            lib().dfft_destroy(self.handle)
            self.handle = None


def fft_mpi_plan_dft_c2c_3d(n0, n1, n2, in_ptr, out_ptr, comm, devIdx, totalDevCount, direction, precision=DOUBLE, flags=0):
    """fft_mpi_plan_dft_c2c_3d (fft_mpi_3d_api.cpp:41-141). `comm` is a LocalComm/BootstrapComm (None for 1 device);
    the `node_data` array of the reference is owned by the communicator here."""
    h = ctypes.c_void_p()
    ch = comm.handle if comm is not None else None
    _check(lib().dfft_plan_c2c_3d(n0, n1, n2, in_ptr, out_ptr, ch, devIdx, totalDevCount, direction, precision, flags, ctypes.byref(h)),
           "fft_mpi_plan_dft_c2c_3d")
    return Plan(h)


def fft_mpi_execute_dft_3d_c2c(plan: Plan):
    plan.execute()


def fft_mpi_destroy_plan(plan: Plan):
    plan.destroy()


def memcpy_htod(dev_ptr, host_ptr, nbytes):
    _check(lib().dfft_memcpy(dev_ptr, host_ptr, nbytes, 1), "dfft_memcpy")


def memcpy_dtoh(host_ptr, dev_ptr, nbytes):
    _check(lib().dfft_memcpy(host_ptr, dev_ptr, nbytes, 2), "dfft_memcpy")


class LinesPlan:
    """templateFFT engine surface (templateFFT.h:361-365): initializeFFT -> LinesPlan(...), launchFFTKernel -> execute,
    deleteFFT -> destroy.  Batched 1-D lines (contiguous or strided) or, with `two_d=(nx, ny, batch)`, batched 2-D."""

    def __init__(self, n=None, stride=1, nlines=0, inner=0, inner_dist=0, outer_dist=0, precision=DOUBLE, two_d=None):
        h = ctypes.c_void_p()
        if two_d is not None:
            _check(lib().dfft_lines_plan_create_2d(two_d[0], two_d[1], two_d[2], precision, ctypes.byref(h)), "dfft_lines_plan_create_2d")
        else:
            _check(lib().dfft_lines_plan_create(n, stride, nlines, inner, inner_dist, outer_dist, precision, ctypes.byref(h)), "dfft_lines_plan_create")
        self.handle = h

    def execute(self, ptr, direction):
        _check(lib().dfft_lines_execute(self.handle, ptr, direction), "dfft_lines_execute")

    def synchronize(self):
        _check(lib().dfft_lines_synchronize(self.handle), "dfft_lines_synchronize")

    @property
    def stream(self):
        return lib().dfft_lines_stream(self.handle)

    def destroy(self):
        if self.handle:
            lib().dfft_lines_destroy(self.handle)
            self.handle = None


def lines_ops(n, stride, nlines, inner, inner_dist, outer_dist, direction, precision=DOUBLE, two_d=False):
    """passes a lines plan would launch (host-only test hook, see dfft_debug_lines_ops)"""
    import json
    need = lib().dfft_debug_lines_ops(n, stride, nlines, inner, inner_dist, outer_dist, precision, direction, int(two_d), None, 0)
    if need < 0:
        raise DfftError("dfft_debug_lines_ops: " + lib().dfft_last_error().decode())
    buf = ctypes.create_string_buffer(int(need))
    lib().dfft_debug_lines_ops(n, stride, nlines, inner, inner_dist, outer_dist, precision, direction, int(two_d), buf, need)
    return json.loads(buf.value.decode())


def fft_lines(ptr, n, stride, nlines, inner, inner_dist, outer_dist, direction, precision=DOUBLE):
    _check(lib().dfft_fft_lines(ptr, n, stride, nlines, inner, inner_dist, outer_dist, direction, precision), "dfft_fft_lines")
