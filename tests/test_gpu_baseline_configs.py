"""BASELINE.json configs at FULL size against the CPU oracle (`-m gpu`; a case is skipped when the box has fewer GPUs):
  C2 512^3 double, 1 GPU          C3 512^3 double, 4 GPUs
  C4 1024^3 double, 8 GPUs        C5 768^3 single, 8 GPUs (mixed radix)
For every config the WHOLE forward spectrum of every device (its transposed y-slab [y_l][z][x]) is compared with the
oracle's slab pipeline on the same heFFTe-test input (std::minstd_rand(4242) -> U(0,1), test_fft3d.h:19-27), like
heFFTe's own test compares the whole world box (test/test_fft3d.h:99-115); then the backward transform of that
spectrum must return N^3 * input within the reference tolerance (1e-11 double / 5e-4 single, test_common.h:136-140).
The default plan flags are used, i.e. the production path of each device count (P2P exchange, stream-pipelined
forward for P > 1)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import distributedfft_b200 as dfft  # noqa: E402
from oracle import BACKWARD, FORWARD, COracle, NumpySlab, SlabGeometry  # noqa: E402
from gpu_helpers import run_slab  # noqa: E402

CONFIGS = [("C2", 512, 1, dfft.DOUBLE, 0), ("C3", 512, 4, dfft.DOUBLE, 0), ("C3b", 512, 8, dfft.DOUBLE, 0), ("C3c", 512, 2, dfft.DOUBLE, 0),
           # the pipelined schedules at full size, also where they are not the default (kernel chain for the cube)
           ("C3-chain", 512, 4, dfft.DOUBLE, dfft.FORCE_PIPELINE), ("C3c-chain", 512, 2, dfft.DOUBLE, dfft.FORCE_PIPELINE),
           ("C4", 1024, 8, dfft.DOUBLE, 0), ("C5", 768, 8, dfft.FLOAT, 0)]


@pytest.mark.parametrize("name,n,P,precision,flags", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_full_size_forward_spectrum_and_round_trip_vs_oracle(name, n, P, precision, flags):
    if torch.cuda.device_count() < P:
        pytest.skip(f"needs {P} GPUs, box has {torch.cuda.device_count()}")
    co = COracle()
    g = SlabGeometry(n, n, n, P)
    ns = NumpySlab(n, n, n, P)
    a = np.empty(n ** 3, dtype=np.complex128)
    co.fill_minstd(a, 4242)
    A = a.reshape(n, n, n)
    inputs = ns.scatter_input(A)
    b1 = [b.copy() for b in inputs]
    b2 = [np.zeros_like(b) for b in b1]
    co.slab_execute(g, b1, b2, FORWARD)          # oracle: reference stages t0..t3 on P "devices"
    del b1
    cast = (lambda x: x) if precision == dfft.DOUBLE else (lambda x: x.astype(np.complex64))
    res = run_slab(n, n, n, P, FORWARD, [cast(b) for b in inputs], precision=precision, repeat=2, refill=False, flags=flags)
    scale = max(np.abs(r[: g.out_count(q)]).max() for q, r in enumerate(b2))
    tol = 1e-12 * np.log2(float(n) ** 3) if precision == dfft.DOUBLE else 5e-6
    for q in range(P):
        cnt = g.out_count(q)
        err = np.abs(res[q]["buf2"][:cnt] - b2[q][:cnt]).max() / scale
        assert err <= tol, (name, "forward", q, err)
    if P > 1:
        assert res[0]["exchange"] == dfft.EXCHANGE_P2P
    spectra = [r["buf2"] for r in res]
    del res, b2
    back = run_slab(n, n, n, P, BACKWARD, spectra, precision=precision, flags=flags)
    rt_tol = 1e-11 if precision == dfft.DOUBLE else 5e-4
    for p in range(P):
        cnt = g.in_count(p)
        err = np.abs(back[p]["buf2"][:cnt] / float(n) ** 3 - inputs[p][:cnt]).max()
        assert err <= rt_tol, (name, "round trip", p, err)


# ---- past 2^31 elements on one device -------------------------------------------------------------------------------------
import kernel_matrix as km  # noqa: E402

# device memory: the input (transformed in place), the plan's copy of it and its work buffer, plus the reference's chunks
BIG = [pytest.param(dfft.FLOAT, 52, id="f32-2048x1024x1024"), pytest.param(dfft.DOUBLE, 100, id="f64-2048x1024x1024")]


def _dft_matrix(n, k, dev):
    """W[j, m] = exp(-2 pi i (j * k_m mod n) / n): the product reduced in integers so the angle is exact"""
    j = torch.arange(n, dtype=torch.int64, device=dev)[:, None]
    ph = (j * torch.as_tensor(k, dtype=torch.int64, device=dev)[None, :]) % n
    ang = ph.double() * (-2.0 * np.pi / n)
    return torch.polar(torch.ones_like(ang), ang)


@pytest.mark.parametrize("precision,gib", BIG)
def test_single_device_transform_past_2_31_elements(precision, gib):
    """2048 x 1024 x 1024 = 2^31 elements on one device: every element offset past 2^31 must be formed in 64 bits.  The whole
    spectrum is too large for a host reference, so 64 complete output x-lines out[ky][kz][:] (ky, kz in {0, 1, N/2, N-1} and
    4 random values each) are computed directly: T = A[x] @ Wz[:, kz] plane by plane in complex128, then Wy[ky, :] @ T, then
    the 2048-point DFT over x as a matrix product; bound as the matrix cases.  Then the SCALE_BACKWARD round trip within 5e-4."""
    n0, n1, n2 = 2048, 1024, 1024
    N = n0 * n1 * n2
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    free, _ = torch.cuda.mem_get_info(dev)
    if free < gib * (1 << 30):
        pytest.skip(f"needs ~{gib} GiB of free device memory, {free / (1 << 30):.0f} GiB free")
    cdt = torch.complex64 if precision == dfft.FLOAT else torch.complex128

    def make_input():
        gen = torch.Generator(device=dev)
        gen.manual_seed(2031)
        return torch.randn((n0, n1, n2), dtype=cdt, device=dev, generator=gen).mul_(np.sqrt(2.0))   # re, im ~ N(0, 1)

    rng = np.random.default_rng(31)
    ky = sorted({0, 1, n1 // 2, n1 - 1} | set(rng.choice(np.arange(2, n1 // 2), 4, replace=False).tolist()))
    kz = sorted({0, 1, n2 // 2, n2 - 1} | set(rng.choice(np.arange(n2 // 2 + 1, n2 - 1), 4, replace=False).tolist()))
    assert len(ky) == len(kz) == 8
    A = make_input()
    Wz, WyT, Wx = _dft_matrix(n2, kz, dev), _dft_matrix(n1, ky, dev).T.contiguous(), _dft_matrix(n0, list(range(n0)), dev)
    U = torch.empty((n0, len(ky), len(kz)), dtype=torch.complex128, device=dev)
    for x0 in range(0, n0, 64):
        T = A[x0: x0 + 64].to(torch.complex128) @ Wz           # [x][y][kz]
        U[x0: x0 + 64] = WyT @ T                                # [x][ky][kz]
        del T
    ref = torch.einsum("xab,xk->abk", U, Wx).cpu().numpy()     # out[ky][kz][kx]
    del U, Wx
    plan = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, A.data_ptr(), None, None, 0, 1, FORWARD, precision)
    plan.execute()
    plan.synchronize()
    plan.destroy()
    got = A.view(n1, n2, n0)[torch.as_tensor(ky, device=dev)][:, torch.as_tensor(kz, device=dev)].to(torch.complex128).cpu().numpy()
    err = km.check(got, ref, precision, N, "2048x1024x1024 forward, 64 sampled x-lines")
    back = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, A.data_ptr(), None, None, 0, 1, BACKWARD, precision, dfft.SCALE_BACKWARD)
    back.execute()
    back.synchronize()
    back.destroy()
    torch.cuda.synchronize()
    A0 = make_input()
    rt = max(float((A[x0: x0 + 64] - A0[x0: x0 + 64]).abs().max()) for x0 in range(0, n0, 64))
    print(f"\n2^31 elements {km.PREC_NAME[precision]}: forward max|err|/rms {err:.3e} (bound {km.bound(precision, N):.3e}), round trip {rt:.3e}")
    assert rt <= 5e-4, rt
