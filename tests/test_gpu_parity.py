"""GPU parity tests (run with `-m gpu` on a B200): the CUDA path through the C ABI versus the CPU
oracle on the same seeded inputs, the committed golden vectors, and size-independent properties at
the BASELINE sizes.  Tolerances: fp64 relative L-inf 1e-12*log2(N) per axis / 1e-11 absolute round
trip on U(0,1) data (heffte/heffteBenchmark/test/test_common.h:136-140); fp32 5e-4."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import distributedfft_b200 as dfft  # noqa: E402
from oracle import BACKWARD, FORWARD, COracle, NumpySlab, SlabGeometry  # noqa: E402
from gpu_helpers import CDT, run_slab  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def co():
    return COracle()


def _dev_array(a, precision):
    npdt, tdt = CDT[precision]
    return torch.from_numpy(np.ascontiguousarray(a, dtype=npdt)).cuda()


def test_library_loaded_and_gpu_present():
    assert torch.cuda.is_available(), "these tests must run on a CUDA device"
    assert os.path.exists(dfft.LIB_PATH)
    assert dfft.lib().dfft_version() >= 100


def test_golden_vectors_through_cabi():
    """heFFTe pen-and-paper box + 11-point DFT is not a supported length (prime 11) -> the box only:
    sizes 2,3,4 are below the kernel's minimum length except 4; check axis of length 4 and the
    12/6/9-point engines against the same closed forms via numpy instead."""
    with open(os.path.join(HERE, "golden", "heffte_vectors.json")) as f:
        gold = json.load(f)
    shape = tuple(gold["box_shape_c_order"])
    c = lambda v: np.asarray(v)[..., 0] + 1j * np.asarray(v)[..., 1]
    x = c(gold["box_input"]).reshape(shape)
    ref = c(gold["box_fft_dim2_axis0"]).reshape(shape)   # transforms over the size-4 (slowest) axis, stride 6
    t = _dev_array(x.reshape(-1), dfft.DOUBLE)
    dfft.fft_lines(t.data_ptr(), 4, 6, 6, 6, 1, 24, FORWARD)
    got = t.cpu().numpy().reshape(shape)
    assert np.abs(got - ref).max() < 1e-11


@pytest.mark.parametrize("precision", [dfft.DOUBLE, dfft.FLOAT])
def test_every_supported_length_per_axis(co, precision):
    """K1/K2 single-axis parity for every instantiated length, contiguous and strided, fwd + inverse."""
    tol = 1e-12 if precision == dfft.DOUBLE else 2e-6
    rng = np.random.default_rng(7)
    for n in dfft.supported_lengths(precision):
        # contiguous: 37 lines (ragged versus the tile width)
        a = rng.standard_normal((37, n)) + 1j * rng.standard_normal((37, n))
        a = a.astype(CDT[precision][0])
        for direction, sign in ((FORWARD, -1), (BACKWARD, +1)):
            ref = co.fft_axis(a.astype(np.complex128), 1, sign)
            t = _dev_array(a.reshape(-1), precision)
            dfft.fft_lines(t.data_ptr(), n, 1, 37, 37, n, 37 * n, direction, precision)
            got = t.cpu().numpy().reshape(37, n)
            err = np.abs(got - ref).max() / np.abs(ref).max()
            assert err <= tol * max(1.0, np.log2(n)), (n, "contig", direction, err)
        # strided: 3 matrices of n rows x 21 columns (21 is ragged for every tile width)
        b = rng.standard_normal((3, n, 21)) + 1j * rng.standard_normal((3, n, 21))
        b = b.astype(CDT[precision][0])
        for direction, sign in ((FORWARD, -1), (BACKWARD, +1)):
            ref = co.fft_axis(b.astype(np.complex128), 1, sign)
            t = _dev_array(b.reshape(-1), precision)
            dfft.fft_lines(t.data_ptr(), n, 21, 3 * 21, 21, 1, n * 21, direction, precision)
            got = t.cpu().numpy().reshape(3, n, 21)
            err = np.abs(got - ref).max() / np.abs(ref).max()
            assert err <= tol * max(1.0, np.log2(n)), (n, "strided", direction, err)


SHAPES_1GPU = [(64, 64, 64), (8, 16, 32), (12, 10, 24), (96, 48, 64), (128, 100, 6), (9, 125, 49)]


@pytest.mark.parametrize("n0,n1,n2", SHAPES_1GPU)
def test_single_gpu_forward_backward_vs_oracle(co, n0, n1, n2):
    """BASELINE config class 2 (1 GPU, no all-to-all) on oracle-sized cubes: forward output layout
    [y][z][x] and values equal the oracle's; backward returns N^3 * input (unnormalised)."""
    rng = np.random.default_rng(n0 * 7 + n1)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    g = SlabGeometry(n0, n1, n2, 1)
    b1 = [A.reshape(-1).copy()]; b2 = [np.zeros_like(b1[0])]
    co.slab_execute(g, b1, b2, FORWARD)
    res = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)])
    scale = np.abs(b2[0]).max()
    assert np.abs(res[0]["buf2"] - b2[0]).max() <= 1e-12 * np.log2(n0 * n1 * n2) * scale
    assert res[0]["launches"] == 3
    # backward from the oracle's forward output
    c1 = [b2[0].copy()]; c2 = [np.zeros_like(c1[0])]
    co.slab_execute(g, c1, c2, BACKWARD)
    resb = run_slab(n0, n1, n2, 1, BACKWARD, [b2[0]])
    assert np.abs(resb[0]["buf2"] - c2[0]).max() <= 1e-12 * np.log2(n0 * n1 * n2) * np.abs(c2[0]).max()
    assert np.abs(resb[0]["buf2"] / (n0 * n1 * n2) - A.reshape(-1)).max() <= 1e-11


def test_single_gpu_float32(co):
    n0, n1, n2 = 48, 96, 64
    rng = np.random.default_rng(5)
    A = (rng.random((n0, n1, n2)) + 1j * rng.random((n0, n1, n2))).astype(np.complex64)
    ref = np.fft.fftn(A.astype(np.complex128)).transpose(1, 2, 0).reshape(-1)
    res = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], precision=dfft.FLOAT)
    assert np.abs(res[0]["buf2"] - ref).max() / np.abs(ref).max() <= 5e-6
    back = run_slab(n0, n1, n2, 1, BACKWARD, [res[0]["buf2"]], precision=dfft.FLOAT)
    assert np.abs(back[0]["buf2"] / (n0 * n1 * n2) - A.reshape(-1)).max() <= 5e-4


def test_inplace_and_scale_flag(co):
    n0, n1, n2 = 32, 16, 64
    rng = np.random.default_rng(3)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    ref = np.fft.fftn(A).transpose(1, 2, 0).reshape(-1)
    res = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], inplace=True)
    assert np.abs(res[0]["buf2"] - ref).max() <= 1e-11 * np.abs(ref).max()
    back = run_slab(n0, n1, n2, 1, BACKWARD, [ref], flags=dfft.SCALE_BACKWARD)
    assert np.abs(back[0]["buf2"] - A.reshape(-1)).max() <= 1e-12


@pytest.mark.parametrize("n0,n1,n2", [(16, 8, 32), (12, 10, 24)])
def test_staged_mode_matches_reference_stage_boundaries(co, n0, n1, n2):
    """dfft_execute_stage leaves bufferDev1/2 as the reference leaves them after t0,t1,t2,t3."""
    rng = np.random.default_rng(11)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    g = SlabGeometry(n0, n1, n2, 1)
    res = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], flags=dfft.EXCHANGE_STAGED, stages=[0, 1, 2, 3])
    for s in range(4):
        o1 = [A.reshape(-1).copy()]; o2 = [np.zeros_like(o1[0])]
        co.slab_execute(g, o1, o2, FORWARD, s)
        d1, d2 = res[0]["stages"][s]
        scale = max(np.abs(o1[0]).max(), 1.0)
        assert np.abs(d1 - o1[0]).max() <= 1e-12 * 12 * scale, s
        if s >= 1:
            assert np.abs(d2 - o2[0]).max() <= 1e-12 * 12 * scale, s


def test_plan_semantics_snapshot_and_reexecute():
    """Plan creation snapshots `in` into bufferDev1 (api.cpp:77) and execute never re-reads `in`.
    Unlike the reference (whose t0 overwrites bufferDev1, so its driver refills it,
    fftSpeed3d_c2c.cpp:78) the fused path leaves bufferDev1 intact: repeated executes give the same
    spectrum, which is what lets bench.py time K identical steps."""
    n = 16
    rng = np.random.default_rng(2)
    A = rng.standard_normal((n, n, n)) + 1j * rng.standard_normal((n, n, n))
    ref = np.fft.fftn(A).transpose(1, 2, 0).reshape(-1)
    res = run_slab(n, n, n, 1, FORWARD, [A.reshape(-1)], repeat=3, refill=False)
    assert np.abs(res[0]["buf2"] - ref).max() <= 1e-11 * np.abs(ref).max()
    assert np.array_equal(res[0]["buf1"], A.reshape(-1))
    t = res[0]["timings"]
    assert len(t) == 5 and t[1] == 0.0 and abs(t[4] - (t[0] + t[2] + t[3])) < 1e-9


def test_error_behaviour():
    with pytest.raises(dfft.DfftError):
        dfft.fft_mpi_plan_dft_c2c_3d(17, 16, 16, 1, 2, None, 0, 1, FORWARD)      # unsupported length
    with pytest.raises(dfft.DfftError):
        dfft.fft_mpi_plan_dft_c2c_3d(16, 16, 16, 1, 2, None, 0, 1, 5)            # bad direction
    with pytest.raises(dfft.DfftError):
        dfft.fft_mpi_plan_dft_c2c_3d(16, 16, 16, 1, 2, None, 0, 2, FORWARD)      # P=2 without a communicator
    with pytest.raises(dfft.DfftError):
        dfft.fft_mpi_alloc_local_memory(16, 7)                                    # bad flag ("Fail to allocate memory!")


def test_baseline_512_cube_properties_and_roundtrip(co):
    """BASELINE config 2 at full size (512^3 double, 1 GPU): driver ramp input round trip with the
    driver's metric (fftSpeed3d_c2c.cpp:61-63, 84-91) <= 1e-11, Parseval, and the spectrum of the
    ramp's DC/plane structure; plus exact comparison of 4 output y-planes with the oracle's 1-D engine."""
    n = 512
    n3 = n ** 3
    cdt = torch.complex128
    dev = torch.device("cuda", 0)
    idx = torch.arange(n3, dtype=torch.float64, device=dev)
    tin = torch.complex(idx, idx)
    del idx
    tout = torch.empty(n3, dtype=cdt, device=dev)
    plan = dfft.fft_mpi_plan_dft_c2c_3d(n, n, n, tin.data_ptr(), tout.data_ptr(), None, 0, 1, FORWARD)
    plan.execute(); plan.synchronize()
    t = plan.timings()
    # Parseval: sum |X|^2 = N^3 sum |x|^2
    e_in = float((tin.real.double() ** 2 + tin.imag.double() ** 2).sum())
    e_out = float((tout.real ** 2 + tout.imag ** 2).sum())
    assert abs(e_out / (n3 * e_in) - 1.0) < 1e-12
    # DC bin = sum of inputs = (1+i) * n3 (n3-1)/2 ; forward output layout [y][z][x]
    dc = complex(tout[0].item())
    exact = n3 * (n3 - 1) / 2
    assert abs(dc.real - exact) / exact < 1e-13 and abs(dc.imag - exact) / exact < 1e-13
    # ramp separability: X[kx,0,0] (x line of y=z=0) = n^2 * n^2 * DFT_n(ramp_x) for kx != 0
    line = tout[:n].cpu().numpy()
    kx = np.arange(1, n)
    expect = (1 + 1j) * (n * n) * (n * n) * (-n / 2 + 0.5j * n / np.tan(np.pi * kx / n))
    assert np.abs(line[1:] - expect).max() / np.abs(expect).max() < 1e-11
    planb = dfft.fft_mpi_plan_dft_c2c_3d(n, n, n, tout.data_ptr(), tin.data_ptr(), None, 0, 1, BACKWARD)
    planb.execute(); planb.synchronize()
    idx = torch.arange(n3, dtype=torch.float64, device=dev)
    er = (tin.real / n3 - idx).abs().max().item()
    ei = (tin.imag / n3 - idx).abs().max().item()
    drv_metric = np.hypot(er, ei) / 1e7
    assert drv_metric <= 1e-11, drv_metric
    plan.destroy(); planb.destroy()
    assert t[4] > 0


@pytest.mark.parametrize("n,n0", [(64, 48), (512, 24), (96, 6), (256, 4), (10, 32), (1024, 6)])
def test_fused_t0_is_bitwise_the_two_sweep_t0(n, n0):
    """The fused persistent t0 kernel (Z and Y roles, intermediate in L2, per-plane completion counters)
    runs the same butterflies in the same order as the two-sweep path: results must be bit-identical,
    forward and backward, over several executes (the counters are monotonic across executes)."""
    rng = np.random.default_rng(n + n0)
    A = rng.standard_normal((n0, n, n)) + 1j * rng.standard_normal((n0, n, n))
    for direction in (FORWARD, BACKWARD):
        inp = A.reshape(-1) if direction == FORWARD else A.transpose(1, 2, 0).reshape(-1)
        a = run_slab(n0, n, n, 1, direction, [inp], repeat=3, refill=False, flags=dfft.FORCE_FUSE)
        b = run_slab(n0, n, n, 1, direction, [inp], repeat=3, refill=False, flags=dfft.NO_FUSE | dfft.NO_TMA)   # same kernels as the fused roles
        assert a[0]["fused"] and not b[0]["fused"]
        assert a[0]["launches"] == 2 and b[0]["launches"] == 3
        assert np.array_equal(a[0]["buf2"], b[0]["buf2"]), (n, n0, direction)
    ref = np.fft.fftn(A).transpose(1, 2, 0).reshape(-1)
    f = run_slab(n0, n, n, 1, FORWARD, [A.reshape(-1)], flags=dfft.FORCE_FUSE)
    assert np.abs(f[0]["buf2"] - ref).max() <= 1e-12 * np.log2(A.size) * np.abs(ref).max()


@pytest.mark.parametrize("n0,n1,n2,precision", [(512, 512, 16, dfft.DOUBLE), (16, 512, 512, dfft.DOUBLE), (24, 1024, 1024, dfft.DOUBLE), (256, 256, 256, dfft.DOUBLE),
                                                 (8, 768, 768, dfft.DOUBLE), (512, 32, 512, dfft.FLOAT), (16, 1024, 1024, dfft.FLOAT), (768, 768, 16, dfft.FLOAT)])
def test_tma_pipelined_passes_match_the_register_staged_kernels(n0, n1, n2, precision):
    """The TMA-ring pass kernels (fft_tma.cuh: Z, natural Y, X with the fused transpose, forward and backward) against the
    register-staged fft_tile_kernel on the same data -- bit for bit where both use the same radix schedule (512: 8.8.8),
    to rounding otherwise -- and against numpy.  Shapes mix axes with and without a TMA instantiation."""
    rng = np.random.default_rng(n0 + n1 + n2)
    npdt = CDT[precision][0]
    A = (rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))).astype(npdt)
    ref = np.fft.fftn(A.astype(np.complex128)).transpose(1, 2, 0).reshape(-1)
    tol = 1e-12 * np.log2(A.size) if precision == dfft.DOUBLE else 5e-6
    a = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], precision=precision, repeat=2, refill=False)
    b = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], precision=precision, flags=dfft.NO_TMA)
    assert np.abs(a[0]["buf2"] - ref).max() <= tol * np.abs(ref).max()
    assert np.abs(a[0]["buf2"] - b[0]["buf2"]).max() <= tol * np.abs(ref).max()
    if precision == dfft.DOUBLE and {n0, n1, n2} <= {512, 16}:
        assert np.array_equal(a[0]["buf2"], b[0]["buf2"])
    spec = a[0]["buf2"]
    ba = run_slab(n0, n1, n2, 1, BACKWARD, [spec], precision=precision, flags=dfft.SCALE_BACKWARD)
    bb = run_slab(n0, n1, n2, 1, BACKWARD, [spec], precision=precision, flags=dfft.SCALE_BACKWARD | dfft.NO_TMA)
    rt = 1e-11 if precision == dfft.DOUBLE else 5e-4
    assert np.abs(ba[0]["buf2"] - A.reshape(-1)).max() <= rt
    assert np.abs(ba[0]["buf2"] - bb[0]["buf2"]).max() <= rt


def test_host_buffer_entry_points_two_plans_in_flight():
    """dfft_execute_host (synchronous) and dfft_execute_host_async with two plans driven alternately
    (what bench.py's e2e leg does): every step's pinned host output equals numpy's fftn of its input."""
    import ctypes
    n0, n1, n2 = 32, 16, 64
    cnt = n0 * n1 * n2
    rng = np.random.default_rng(21)
    xs = [rng.standard_normal(cnt) + 1j * rng.standard_normal(cnt) for _ in range(2)]
    refs = [np.fft.fftn(x.reshape(n0, n1, n2)).transpose(1, 2, 0).reshape(-1) for x in xs]
    dev = torch.device("cuda", 0)
    bufs = [torch.zeros(cnt, dtype=torch.complex128, device=dev) for _ in range(2)]
    plans = [dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, b.data_ptr(), None, None, 0, 1, FORWARD) for b in bufs]
    hin = [dfft.fft_mpi_alloc_local_memory(cnt, dfft.ALLOC_CPU) for _ in range(2)]
    hout = [dfft.fft_mpi_alloc_local_memory(cnt, dfft.ALLOC_CPU) for _ in range(2)]
    for k in range(2):
        ctypes.memmove(hin[k], xs[k].ctypes.data, cnt * 16)
    plans[0].execute_host(hin[0], hout[0])
    got = np.empty(cnt, dtype=np.complex128)
    ctypes.memmove(got.ctypes.data, hout[0], cnt * 16)
    assert np.abs(got - refs[0]).max() <= 1e-11 * np.abs(refs[0]).max()
    ctypes.memset(hout[0], 0, cnt * 16)
    for it in range(6):
        plans[it % 2].execute_host_async(hin[it % 2], hout[it % 2])
    for k in range(2):
        plans[k].synchronize()
        ctypes.memmove(got.ctypes.data, hout[k], cnt * 16)
        assert np.abs(got - refs[k]).max() <= 1e-11 * np.abs(refs[k]).max()
    for k in range(2):
        plans[k].destroy()
        dfft.lib().dfft_free_local(hin[k], dfft.ALLOC_CPU)
        dfft.lib().dfft_free_local(hout[k], dfft.ALLOC_CPU)


GENERIC_LENGTHS = [2, 3, 5, 7, 11, 13, 15, 30, 77, 143, 360, 1001, 2187, 3000, 3125, 6400]


@pytest.mark.parametrize("precision", [dfft.DOUBLE, dfft.FLOAT])
def test_generic_lengths_per_axis(co, precision):
    """Lengths without a tuned kernel run on the run-time-scheduled kernel (fft_generic.cuh): every
    2..13-smooth length the reference's generator accepts (templateFFT.cpp:3956-3964), contiguous and
    strided, forward and inverse, against numpy's pocketfft."""
    tol = 1e-12 if precision == dfft.DOUBLE else 3e-6
    rng = np.random.default_rng(17)
    for n in GENERIC_LENGTHS:
        assert dfft.length_kind(n, precision) == 1, n
        a = (rng.standard_normal((5, n)) + 1j * rng.standard_normal((5, n))).astype(CDT[precision][0])
        b = (rng.standard_normal((2, n, 11)) + 1j * rng.standard_normal((2, n, 11))).astype(CDT[precision][0])
        for direction in (FORWARD, BACKWARD):
            f = np.fft.fft if direction == FORWARD else (lambda x, axis: np.fft.ifft(x, axis=axis) * x.shape[axis])
            ref = f(a.astype(np.complex128), axis=1)
            t = _dev_array(a.reshape(-1), precision)
            dfft.fft_lines(t.data_ptr(), n, 1, 5, 5, n, 5 * n, direction, precision)
            err = np.abs(t.cpu().numpy().reshape(5, n) - ref).max() / np.abs(ref).max()
            assert err <= tol * max(1.0, np.log2(n)), (n, "contig", direction, err)
            ref = f(b.astype(np.complex128), axis=1)
            t = _dev_array(b.reshape(-1), precision)
            dfft.fft_lines(t.data_ptr(), n, 11, 2 * 11, 11, 1, n * 11, direction, precision)
            err = np.abs(t.cpu().numpy().reshape(2, n, 11) - ref).max() / np.abs(ref).max()
            assert err <= tol * max(1.0, np.log2(n)), (n, "strided", direction, err)
    assert dfft.length_kind(17, precision) == 0 and dfft.length_kind(6561 * 2, precision) == 0


def test_golden_11_point_dft_and_box_all_axes():
    """The reference tree's pen-and-paper vectors through the C ABI: 11-point DFT of 1..11
    (test_units_stock.cpp:229-255) and the 2x3x4 box along every axis (test_units_nompi.cpp:136-190)."""
    with open(os.path.join(HERE, "golden", "heffte_vectors.json")) as f:
        gold = json.load(f)
    c = lambda v: np.asarray(v)[..., 0] + 1j * np.asarray(v)[..., 1]
    x11 = np.arange(1, 12, dtype=np.complex128)
    t = _dev_array(x11, dfft.DOUBLE)
    dfft.fft_lines(t.data_ptr(), 11, 1, 1, 1, 11, 11, FORWARD)
    assert np.abs(c(gold["dft11_input"]).reshape(-1) - x11).max() == 0
    assert np.abs(t.cpu().numpy() - c(gold["dft11_output"]).reshape(-1)).max() < 1e-11
    shape = tuple(gold["box_shape_c_order"])   # (4, 3, 2): axis 2 fastest
    x = c(gold["box_input"]).reshape(shape)
    # axis 2 (length 2, contiguous), axis 1 (length 3, stride 2), axis 0 (length 4, stride 6)
    for key, n, stride, nlines, inner, inner_dist, outer in (("box_fft_dim0_axis2", 2, 1, 12, 12, 2, 24),
                                                           ("box_fft_dim1_axis1", 3, 2, 8, 2, 1, 6),
                                                           ("box_fft_dim2_axis0", 4, 6, 6, 6, 1, 24)):
        t = _dev_array(x.reshape(-1), dfft.DOUBLE)
        dfft.fft_lines(t.data_ptr(), n, stride, nlines, inner, inner_dist, outer, FORWARD)
        assert np.abs(t.cpu().numpy().reshape(shape) - c(gold[key]).reshape(shape)).max() < 1e-11, key


@pytest.mark.parametrize("n0,n1,n2", [(15, 22, 26), (6, 35, 33), (64, 64, 64)])
def test_generic_kernel_3d_forward_backward(co, n0, n1, n2, monkeypatch):
    """Whole slab path on the run-time-scheduled kernel: lengths without tuned kernels, and (DFFT_GENERIC=1) the
    generic kernel on a tuned size must agree with the tuned kernels to rounding."""
    rng = np.random.default_rng(n0 + n1)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    ref = np.fft.fftn(A).transpose(1, 2, 0).reshape(-1)
    if (n0, n1, n2) == (64, 64, 64):
        monkeypatch.setenv("DFFT_GENERIC", "1")
    res = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)])
    assert np.abs(res[0]["buf2"] - ref).max() <= 1e-12 * np.log2(A.size) * np.abs(ref).max()
    back = run_slab(n0, n1, n2, 1, BACKWARD, [ref])
    assert np.abs(back[0]["buf2"] / A.size - A.reshape(-1)).max() <= 1e-11


def test_lines_plan_2d_and_reuse():
    """The engine surface (initializeFFT / launchFFTKernel / deleteFFT -> LinesPlan): a batched 2-D plan reused for
    several launches, forward then inverse, against numpy's fft2."""
    nx, ny, batch = 64, 48, 5
    rng = np.random.default_rng(4)
    a = rng.standard_normal((batch, ny, nx)) + 1j * rng.standard_normal((batch, ny, nx))
    ref = np.fft.fft2(a, axes=(1, 2))
    plan = dfft.LinesPlan(two_d=(nx, ny, batch))
    t = _dev_array(a.reshape(-1), dfft.DOUBLE)
    plan.execute(t.data_ptr(), FORWARD); plan.synchronize()
    assert np.abs(t.cpu().numpy().reshape(batch, ny, nx) - ref).max() <= 1e-12 * 12 * np.abs(ref).max()
    plan.execute(t.data_ptr(), BACKWARD); plan.synchronize()
    assert np.abs(t.cpu().numpy().reshape(batch, ny, nx) / (nx * ny) - a).max() <= 1e-12
    t2 = _dev_array(a.reshape(-1), dfft.DOUBLE)
    plan.execute(t2.data_ptr(), FORWARD); plan.synchronize()
    assert np.abs(t2.cpu().numpy().reshape(batch, ny, nx) - ref).max() <= 1e-12 * 12 * np.abs(ref).max()
    plan.destroy()


def test_batch_benchmark_driver_surface(tmp_path):
    """batchFFT 1d|2d X Y Z num_iter printResult: stdout lines and CSV columns of templateFFT/batchTest/Test_1D.cpp:139-176
    and Test_2D.cpp (runTest1D_opt.sh:4 header), round-trip error on the ramp input."""
    import re
    import subprocess
    exe = os.path.join(os.path.dirname(HERE), "distributedfft_b200", "batchFFT")
    assert os.path.exists(exe), "batchFFT was not built"
    for mode, args, dims in (("1d", ["1024", "1", "1"], "1024x65536x1"), ("2d", ["256", "128", "1"], "256x128x2048")):
        csv = tmp_path / f"batch_{mode}.csv"
        r = subprocess.run([exe, mode] + args + ["3", "1", str(csv)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        assert f"1 - FFT + iFFT C2C {mode.upper()} in double precision LUT" in r.stdout
        m = re.search(r"FFT: (\S+) Buffer: ([0-9.]+) MB avg_hip_time: ([0-9.]+) ms Gflops: ([0-9.]+) num_iter: 3", r.stdout)
        assert m and m.group(1) == dims and float(m.group(2)) == 1024.0, r.stdout
        err = float(re.search(r"Max error: (\S+)", r.stdout).group(1))
        assert err < 1e-6      # ramp values reach 6.7e7; the reference prints 3.5e-13..6.7e-11 relative to far smaller batches
        assert "element 0 input:  (1,0)" in r.stdout
        cols = csv.read_text().strip().split(",")
        assert len(cols) == 9 and cols[0] == args[0]


def test_compute_sanitizer_memcheck_and_racecheck():
    """SURVEY appendix D: the driver on a small cube under compute-sanitizer (memcheck, racecheck) is clean."""
    import shutil
    import subprocess
    cs = shutil.which("compute-sanitizer") or "/usr/local/cuda/bin/compute-sanitizer"
    if not os.path.exists(cs):
        pytest.skip("compute-sanitizer not installed")
    exe = os.path.join(os.path.dirname(HERE), "distributedfft_b200", "distFFT")
    for tool in ("memcheck", "racecheck"):
        r = subprocess.run([cs, "--tool", tool, "--error-exitcode", "7", exe, "16", "16", "16", "1"], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (tool, r.stdout[-3000:], r.stderr[-2000:])
        assert "ERROR SUMMARY: 0 errors" in r.stdout or "RACECHECK SUMMARY: 0 hazards" in r.stdout, (tool, r.stdout[-1500:])


@pytest.mark.parametrize("precision", [dfft.DOUBLE, dfft.FLOAT])
def test_four_step_long_lines(precision):
    """Lines longer than one shared-memory line go through the two-pass four-step plan: the lengths the reference's
    Test_1D sweep reaches with multi-upload axes (templateFFT.cpp:4007-4106, runTest1D_opt.sh:5-21)."""
    tol = 1e-12 if precision == dfft.DOUBLE else 5e-6
    rng = np.random.default_rng(23)
    for n in (8192, 16384, 131072, 6561, 19683, 78125, 16807, 12000):
        a = (rng.standard_normal((3, n)) + 1j * rng.standard_normal((3, n))).astype(CDT[precision][0])
        plan = dfft.LinesPlan(n, 1, 3, 3, n, 0, precision)
        for direction in (FORWARD, BACKWARD):
            ref = np.fft.fft(a.astype(np.complex128), axis=1) if direction == FORWARD else np.fft.ifft(a.astype(np.complex128), axis=1) * n
            t = _dev_array(a.reshape(-1), precision)
            plan.execute(t.data_ptr(), direction); plan.synchronize()
            err = np.abs(t.cpu().numpy().reshape(3, n) - ref).max() / np.abs(ref).max()
            assert err <= tol * np.log2(n), (n, direction, err)
        plan.destroy()


@pytest.mark.parametrize("n0,n1,n2", [(16, 32, 8), (48, 64, 64), (15, 22, 26)])
def test_natural_order_spectrum_single_device(n0, n1, n2):
    """DFFT_NATURAL_SPECTRUM: forward output / backward input in natural [x][y][z] order (SURVEY 8f rank 1)."""
    rng = np.random.default_rng(n0 + n2)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    ref = np.fft.fftn(A).reshape(-1)
    f = run_slab(n0, n1, n2, 1, FORWARD, [A.reshape(-1)], flags=dfft.NATURAL_SPECTRUM)
    assert np.abs(f[0]["buf2"] - ref).max() <= 1e-12 * np.log2(A.size) * np.abs(ref).max()
    b = run_slab(n0, n1, n2, 1, BACKWARD, [ref], flags=dfft.NATURAL_SPECTRUM)
    assert np.abs(b[0]["buf2"] / A.size - A.reshape(-1)).max() <= 1e-11


# ---- the instantiation matrix (tests/kernel_matrix.py): every kernel the library ships, against an fp64 reference ----------
import kernel_matrix as km  # noqa: E402
from gpu_helpers import run_matrix_case  # noqa: E402

MATRIX_1 = km.single_device_cases()


@pytest.mark.parametrize("case", MATRIX_1, ids=[c.id for c in MATRIX_1])
def test_kernel_matrix_single_device(case, monkeypatch):
    """One tuned length (or generic / TMA configuration) per case: forward and backward against numpy's fftn in complex128 of the
    same rounded input, max|err| / rms(ref) <= 1e-13 log2 N (fp64) / 1e-6 log2 N (fp32), plus the SCALE_BACKWARD round trip; the
    plan must report the path the case names (fused, TMA mask)."""
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    run_matrix_case(case)


FOUR_STEP_CASES = [(p, first, n) for p in (km.D, km.F) for t in (km.FOUR_STEP[p], km.FOUR_STEP_GENERIC[p]) for first, n in t.items()]


@pytest.mark.parametrize("precision,first,n", FOUR_STEP_CASES, ids=[f"{km.PREC_NAME[p]}-{n}-first{f}" for p, f, n in FOUR_STEP_CASES])
def test_kernel_matrix_four_step(precision, first, n):
    """Long lines through the four-step plan, whose first pass (PK_XF_TW of the first factor) runs every tuned length."""
    nl = km.four_step_lines(n)
    rng = np.random.default_rng(n)
    a = (rng.standard_normal((nl, n)) + 1j * rng.standard_normal((nl, n))).astype(CDT[precision][0])
    plan = dfft.LinesPlan(n, 1, nl, nl, n, 0, precision)
    try:
        for direction in (FORWARD, BACKWARD):
            ref = np.fft.fft(a.astype(np.complex128), axis=1) if direction == FORWARD else np.fft.ifft(a.astype(np.complex128), axis=1) * n
            t = _dev_array(a.reshape(-1), precision)
            plan.execute(t.data_ptr(), direction)
            plan.synchronize()
            km.check(t.cpu().numpy(), ref, precision, n, f"four-step {n} = {first} x {n // first} direction {direction}")
    finally:
        plan.destroy()
