"""Helpers for the -m gpu parity tests: drive libdfft.so through its C ABI (via the ctypes
binding) on torch-allocated device buffers, one host thread per device like the reference driver
(3dmpifft_opt/fftSpeed3d_c2c.cpp:49-51)."""
import functools
import threading

import numpy as np
import torch

import distributedfft_b200 as dfft
import kernel_matrix as km
from oracle import NumpySlab, SlabGeometry

CDT = {dfft.DOUBLE: (np.complex128, torch.complex128), dfft.FLOAT: (np.complex64, torch.complex64)}


def run_slab(n0, n1, n2, P, direction, inputs, precision=dfft.DOUBLE, flags=0, repeat=1, stages=None, inplace=False, refill=True):
    """inputs[p]: numpy array (max_count) for device p's bufferDev1.  Returns dict with per-device
    'buf1', 'buf2' numpy copies after execution (and after each stage when `stages`)."""
    g = SlabGeometry(n0, n1, n2, P)
    npdt, tdt = CDT[precision]
    comm = dfft.LocalComm(P) if P > 1 else None
    res = [None] * P
    errs = []

    def worker(p):
        try:
            torch.cuda.set_device(p)
            dev = torch.device("cuda", p)
            mc = g.max_count(p)
            tin = torch.zeros(mc, dtype=tdt, device=dev)
            tin[: inputs[p].size] = torch.from_numpy(np.ascontiguousarray(inputs[p], dtype=npdt)).to(dev)
            tout = tin if inplace else torch.zeros(mc, dtype=tdt, device=dev)
            torch.cuda.synchronize(dev)
            plan = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, tin.data_ptr(), None if inplace else tout.data_ptr(), comm, p, P,
                                                direction, precision, flags)
            out = {}

            def fetch(ptr, count):
                host = np.empty(count, dtype=npdt)
                dfft.memcpy_dtoh(host.ctypes.data, ptr, host.nbytes)
                return host

            if stages is not None:
                out["stages"] = []
                for s in stages:
                    plan.execute_stage(s)
                    out["stages"].append((fetch(plan.bufferDev1, mc), fetch(plan.bufferDev2, mc)))
            else:
                for _ in range(repeat):
                    if _ > 0 and refill:  # refill bufferDev1 like the reference driver (fftSpeed3d_c2c.cpp:78)
                        plan.synchronize()
                        torch.cuda.synchronize(dev)
                        h = np.zeros(mc, dtype=npdt); h[: inputs[p].size] = inputs[p]
                        dfft.memcpy_htod(plan.bufferDev1, h.ctypes.data, h.nbytes)
                    plan.execute()
                plan.synchronize()
                out["timings"] = plan.timings()
                out["launches"] = plan.launches
                out["exchange"] = plan.exchange
                out["fused"] = plan.fused
                out["tma_mask"] = plan.tma_mask
                out["pipeline_chain"] = plan.pipeline_chain
            out["buf1"] = fetch(plan.bufferDev1, mc)
            out["buf2"] = fetch(plan.bufferDev2, mc)
            out["counts"] = (plan.in_count, plan.out_count, plan.maxDataCountInDevice)
            plan.destroy()
            res[p] = out
        except Exception as exc:  # noqa
            import traceback
            errs.append((p, traceback.format_exc()))

    if P == 1:
        worker(0)
    else:
        th = [threading.Thread(target=worker, args=(p,)) for p in range(P)]
        for t in th: t.start()
        for t in th: t.join()
    if comm is not None:
        comm.destroy()
    if errs:
        raise RuntimeError("device thread failed:\n" + "\n".join(e for _, e in errs))
    return res


@functools.lru_cache(maxsize=1)
def matrix_data(shape, precision):
    """seeded standard-normal complex input A [x][y][z] and backward input B [y][z][x], both rounded to `precision`, and
    their fp64 references: the forward spectrum of A laid out [y][z][x], the unnormalised inverse of B laid out [x][y][z]"""
    n0, n1, n2 = shape
    npdt = CDT[precision][0]
    rng = np.random.default_rng([n0, n1, n2, precision])
    A = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(npdt)
    B = (rng.standard_normal((n1, n2, n0)) + 1j * rng.standard_normal((n1, n2, n0))).astype(npdt)
    ref_f = np.ascontiguousarray(np.fft.fftn(A.astype(np.complex128)).transpose(1, 2, 0))
    ref_b = np.fft.ifftn(B.astype(np.complex128).transpose(2, 0, 1)) * (n0 * n1 * n2)
    return A, B, ref_f, ref_b


def run_matrix_case(case):
    """one kernel_matrix case on case.P devices against the fp64 reference (environment already set): forward, backward
    and the scaled round trip, per device over its slab; every plan must have taken the path the case names"""
    n0, n1, n2 = case.shape
    N = n0 * n1 * n2
    P = case.P
    g = SlabGeometry(n0, n1, n2, P)
    A, B, ref_f, ref_b = matrix_data(case.shape, case.precision)

    def expect(res, direction):
        for r in res:
            for k, _ in case.expect:
                v = km.expected(case, k, direction)
                if k == "pipeline_chain" and direction != dfft.FORWARD:
                    continue
                assert r[k] == v, (case.id, direction, k, r[k], v)

    fwd = None
    if dfft.FORWARD in case.directions:
        fwd = run_slab(n0, n1, n2, P, dfft.FORWARD, NumpySlab(n0, n1, n2, P).scatter_input(A), case.precision, case.flags)
        expect(fwd, dfft.FORWARD)
        for q in range(P):
            want = ref_f[q * g.yd: q * g.yd + g.n1l(q)]
            km.check(fwd[q]["buf2"][: g.out_count(q)], want, case.precision, N, f"{case.id} forward device {q}")
    if dfft.BACKWARD in case.directions:
        ins = []
        for q in range(P):
            b = np.zeros(g.max_count(q), dtype=B.dtype)
            blk = B[q * g.yd: q * g.yd + g.n1l(q)].reshape(-1)
            b[: blk.size] = blk
            ins.append(b)
        bwd = run_slab(n0, n1, n2, P, dfft.BACKWARD, ins, case.precision, case.flags)
        expect(bwd, dfft.BACKWARD)
        for p in range(P):
            want = ref_b[p * g.xd: p * g.xd + g.n0l(p)]
            km.check(bwd[p]["buf2"][: g.in_count(p)], want, case.precision, N, f"{case.id} backward device {p}")
        if fwd is not None:
            rt = run_slab(n0, n1, n2, P, dfft.BACKWARD, [r["buf2"] for r in fwd], case.precision, case.flags | dfft.SCALE_BACKWARD)
            expect(rt, dfft.BACKWARD)
            for p in range(P):
                want = A[p * g.xd: p * g.xd + g.n0l(p)]
                km.check(rt[p]["buf2"][: g.in_count(p)], want, case.precision, N, f"{case.id} scaled round trip device {p}")
