"""Multi-GPU parity tests (`-m gpu`; each case is skipped when the box has fewer GPUs than it needs).
P device-threads of one process -- the reference driver's `#pragma omp parallel for num_threads(devices)`
mode (3dmpifft_opt/fftSpeed3d_c2c.cpp:49-51) -- drive libdfft.so through the C ABI; every device's
bufferDev2 is compared with the CPU oracle's P-device restatement of t0..t3
(3dmpifft_opt/include/fft_mpi_3d_api.cpp:181-214, exchange tables :84-133) on the same inputs.
All three exchanges are covered: P2P-fused (Y-pass stores land in the peers' receive buffers over
NVLink), NCCL (grouped send/recv or ncclAlltoAll) and the reference-like staged mode."""
import os
import re
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import distributedfft_b200 as dfft  # noqa: E402
from oracle import BACKWARD, FORWARD, COracle, NumpySlab, SlabGeometry  # noqa: E402
from gpu_helpers import run_slab  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def need(P):
    if torch.cuda.device_count() < P:
        pytest.skip(f"needs {P} GPUs, box has {torch.cuda.device_count()}")


@pytest.fixture(scope="module")
def co():
    return COracle()


MODES = {"p2p": dfft.EXCHANGE_P2P, "nccl": dfft.EXCHANGE_NCCL, "staged": dfft.EXCHANGE_STAGED,
         # the stream-pipelined schedules (z-parts on two streams), forced also where they are not the default
         "p2p-pipe": dfft.EXCHANGE_P2P | dfft.FORCE_PIPELINE, "nccl-pipe": dfft.EXCHANGE_NCCL | dfft.FORCE_PIPELINE,
         "p2p-nopipe": dfft.EXCHANGE_P2P | dfft.NO_PIPELINE}
# (P, n0, n1, n2): even and uneven (short last slab in x and/or y) splits
CASES = [(2, 128, 128, 128), (4, 128, 128, 128), (2, 4, 1024, 1024), (2, 6, 768, 768), (2, 30, 21, 10), (2, 16, 16, 16), (2, 6, 9, 9), (4, 12, 10, 10), (2, 10, 9, 4), (2, 64, 48, 96), (4, 12, 10, 24), (4, 64, 64, 64), (8, 64, 64, 64), (8, 100, 125, 8),
         (8, 24, 48, 16)]


def _oracle(co, g, A, direction):
    ns = NumpySlab(g.n0, g.n1, g.n2, g.P)
    if direction == FORWARD:
        b1 = ns.scatter_input(A)
    else:   # backward input = per-device [y_l][z][x] slabs
        b1 = []
        for q in range(g.P):
            b = np.zeros(g.max_count(q), dtype=np.complex128)
            blk = A[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1)
            b[: blk.size] = blk
            b1.append(b)
    inputs = [b.copy() for b in b1]
    b2 = [np.zeros_like(b) for b in b1]
    co.slab_execute(g, b1, b2, direction)
    return inputs, b2


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("P,n0,n1,n2", CASES)
def test_multi_gpu_forward_backward_vs_oracle(co, mode, P, n0, n1, n2):
    need(P)
    g = SlabGeometry(n0, n1, n2, P)
    rng = np.random.default_rng(n0 * 131 + n1 * 7 + P)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    tol = 1e-12 * np.log2(n0 * n1 * n2)
    for direction in (FORWARD, BACKWARD):
        inputs, ref = _oracle(co, g, A, direction)
        res = run_slab(n0, n1, n2, P, direction, inputs, flags=MODES[mode], repeat=2)
        scale = max(np.abs(r).max() for r in ref)
        for p in range(P):
            n = g.out_count(p) if direction == FORWARD else g.in_count(p)
            err = np.abs(res[p]["buf2"][:n] - ref[p][:n]).max()
            assert err <= tol * scale, (mode, direction, p, err)
            assert res[p]["exchange"] == (MODES[mode] & 3)


@pytest.mark.parametrize("P", [2, 4, 8])
def test_multi_gpu_spectrum_and_round_trip(co, P):
    """Forward spectrum gathered from the y-slabs equals numpy's fftn of the global cube; backward of it
    returns N^3 * input within the reference tolerance 1e-11 (test_common.h:136-140) on U(0,1) data."""
    need(P)
    n0, n1, n2 = 64, 128, 32
    g = SlabGeometry(n0, n1, n2, P)
    ns = NumpySlab(n0, n1, n2, P)
    a = np.zeros(n0 * n1 * n2, dtype=np.complex128)
    co.fill_minstd(a, 4242)
    A = a.reshape(n0, n1, n2)
    res = run_slab(n0, n1, n2, P, FORWARD, ns.scatter_input(A))
    S = ns.gather_forward_output([r["buf2"] for r in res])
    ref = np.fft.fftn(A)
    assert np.abs(S - ref).max() <= 1e-12 * 18 * np.abs(ref).max()
    back = run_slab(n0, n1, n2, P, BACKWARD, [r["buf2"] for r in res])
    B = ns.gather_natural([r["buf2"] for r in back]) / (n0 * n1 * n2)
    assert np.abs(B - A).max() <= 1e-11


@pytest.mark.parametrize("P,n0,n1,n2", [(2, 96, 48, 64), (4, 96, 48, 64), (8, 96, 48, 64), (2, 4, 768, 768), (2, 4, 1024, 1024), (2, 22, 15, 15)])
def test_multi_gpu_float32(P, n0, n1, n2):
    need(P)
    ns = NumpySlab(n0, n1, n2, P)
    rng = np.random.default_rng(P)
    A = (rng.random((n0, n1, n2)) + 1j * rng.random((n0, n1, n2))).astype(np.complex64)
    res = run_slab(n0, n1, n2, P, FORWARD, ns.scatter_input(A), precision=dfft.FLOAT)
    S = ns.gather_forward_output([r["buf2"] for r in res])
    ref = np.fft.fftn(A.astype(np.complex128))
    assert np.abs(S - ref).max() / np.abs(ref).max() <= 5e-6
    back = run_slab(n0, n1, n2, P, BACKWARD, [r["buf2"] for r in res], precision=dfft.FLOAT)
    B = ns.gather_natural([r["buf2"] for r in back]) / (n0 * n1 * n2)
    assert np.abs(B - A).max() <= 5e-4


REPORT = re.compile(
    r"Size:\s+(\d+)x(\d+)x(\d+)\s*\nMPI ranks:\s+(\d+)\s*\nForward FFT time:\s+([0-9.e+-]+) \(s\)\s*\n"
    r"Performance:\s+([0-9.e+-]+) GFlops/s\s*\nMax error:\s+([0-9.e+-]+)")
STAGES = re.compile(r"^t0: [0-9.]+, t1: [0-9.]+, t2: [0-9.]+, t3: [0-9.]+, total: [0-9.]+$", re.M)


@pytest.mark.parametrize("P", [1, 2, 8])
def test_speedtest_driver_report(P):
    """distFFT NX NY NZ GPU_COUNT: the reference driver's stdout surface (fftSpeed3d_c2c.cpp:129-137,
    fft_mpi_3d_api.cpp:201, 270, 285) and its round-trip metric on the ramp input."""
    need(P)
    exe = os.path.join(ROOT, "distributedfft_b200", "distFFT")
    assert os.path.exists(exe), "distFFT driver was not built (python -m distributedfft_b200.build)"
    r = subprocess.run([exe, "64", "64", "64", str(P)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"allocate {P} devices to node 0" in r.stdout
    assert "data count in device 0 of node 0: %d" % (64 ** 3 // P) in r.stdout
    assert len(STAGES.findall(r.stdout)) >= 4 * P      # every device thread prints each forward execute
    m = REPORT.search(r.stdout)
    assert m, r.stdout
    assert m.group(1, 2, 3, 4) == ("64", "64", "64", str(P))
    assert float(m.group(7)) <= 1e-11
    sh = subprocess.run(["bash", os.path.join(ROOT, "distributedfft_b200", "speedTest.sh"), str(P), "16", "16", "16"],
                        capture_output=True, text=True, timeout=120)
    assert sh.returncode == 0 and REPORT.search(sh.stdout), sh.stdout + sh.stderr
    bad = subprocess.run([exe, "64", "64"], capture_output=True, text=True, timeout=60)
    assert bad.returncode != 0 and "The format of arguments should be [NX, NY, NZ, GPU_COUNT]!" in bad.stdout


@pytest.mark.parametrize("P", [2, 4, 8])
def test_baseline_512_cube_multi_gpu_round_trip(P):
    """BASELINE config 3 class at full size (512^3 double over P GPUs): ramp input, driver metric <= 1e-11."""
    need(P)
    exe = os.path.join(ROOT, "distributedfft_b200", "distFFT")
    r = subprocess.run([exe, "512", "512", "512", str(P)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    m = REPORT.search(r.stdout)
    assert m and float(m.group(7)) <= 1e-11, r.stdout[-1500:]


PROC_WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
mode = sys.argv[2]
import numpy as np, torch, torch.distributed as dist
import distributedfft_b200 as dfft
from oracle import NumpySlab, SlabGeometry
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("gloo")
def ag(b):
    out = [None] * world
    dist.all_gather_object(out, b)
    return out
comm = dfft.BootstrapComm(rank, world, ag)
n0, n1, n2 = 48, 64, 32
g = SlabGeometry(n0, n1, n2, world); ns = NumpySlab(n0, n1, n2, world)
rng = np.random.default_rng(99)
A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
ref = np.fft.fftn(A)
mine = ns.scatter_input(A)[rank]
tin = torch.from_numpy(mine).cuda(); tout = torch.zeros_like(tin)
flags = {"p2p": dfft.EXCHANGE_P2P, "nccl": dfft.EXCHANGE_NCCL}[mode]
plan = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, tin.data_ptr(), tout.data_ptr(), comm, rank, world, dfft.FORWARD, dfft.DOUBLE, flags)
for _ in range(3):
    plan.execute()
plan.synchronize()
got = tout.cpu().numpy()[: g.out_count(rank)].reshape(g.n1l(rank), n2, n0)
want = ref[:, rank * g.yd: rank * g.yd + g.n1l(rank), :].transpose(1, 2, 0)
err = np.abs(got - want).max() / np.abs(ref).max()
assert err < 2e-11, err
back = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, tout.data_ptr(), tin.data_ptr(), comm, rank, world, dfft.BACKWARD, dfft.DOUBLE, flags)
back.execute(); back.synchronize()
rt = np.abs(tin.cpu().numpy()[: g.in_count(rank)] / (n0 * n1 * n2) - mine[: g.in_count(rank)]).max()
assert rt < 1e-11, rt
plan.destroy(); back.destroy(); comm.destroy()
dist.barrier(); dist.destroy_process_group()
sys.stdout.write("rank %d ok %s %.2e %.2e\n" % (rank, mode, err, rt)); sys.stdout.flush()
'''


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_process_per_gpu_bootstrap(tmp_path, mode):
    """One process per GPU (torchrun), CUDA-IPC peer mappings / NCCL id swapped through the bootstrap
    all-gather: the launch mode bench.py --gpus N uses."""
    P = 2
    need(P)
    script = tmp_path / "worker.py"
    script.write_text(PROC_WORKER)
    import sys
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={P}", "--master-addr", "127.0.0.1",
                        "--master-port", "29581", str(script), ROOT, mode], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for k in range(P):
        assert f"rank {k} ok" in r.stdout


# the 8-device cases of this EXPERIMENTAL (non-default) kernel have not been on an 8-GPU box yet (none could be had in round 2):
# they stay opt-in so that a surprise there cannot stop `pytest -x` before the product-path tests that sort after this file
NOT_ON_8_YET = pytest.mark.skipif(os.environ.get("DFFT_TEST_EXPERIMENTAL") != "1", reason="experimental kernel, 8-device case not yet run on hardware: set DFFT_TEST_EXPERIMENTAL=1")


@pytest.mark.parametrize("P,n", [(2, 64), (4, 64), pytest.param(8, 64, marks=NOT_ON_8_YET), (2, 128), (2, 256), pytest.param(8, 256, marks=NOT_ON_8_YET)])
def test_overlapped_forward_matches_default_path(P, n):
    """DFFT_OVERLAP_X (fft_fused3_kernel: Z + Y/peer-store + X roles of all z-parts from one ticket stream, per-part arrival
    flags published once per CTA and part) must produce the same y-slabs as the plain P2P path, bit for bit, over repeated
    executes.  Validated on hardware in round 2 (slower than the plain path, DESIGN.md 5.1: kept as an experiment)."""
    need(P)
    n0 = n   # the single-kernel path needs a cube (all three axes share one table entry)
    ns = NumpySlab(n0, n, n, P)
    rng = np.random.default_rng(n + P)
    A = rng.standard_normal((n0, n, n)) + 1j * rng.standard_normal((n0, n, n))
    # the same register-staged kernels on both sides (the TMA X kernel of the default path uses another radix schedule at 256)
    a = run_slab(n0, n, n, P, FORWARD, ns.scatter_input(A), flags=dfft.EXCHANGE_P2P | dfft.NO_TMA | dfft.NO_PIPELINE, repeat=3, refill=False)
    b = run_slab(n0, n, n, P, FORWARD, ns.scatter_input(A), flags=dfft.EXCHANGE_P2P | dfft.OVERLAP_X, repeat=3, refill=False)
    for p in range(P):
        assert b[p]["launches"] < a[p]["launches"]
        assert np.array_equal(a[p]["buf2"], b[p]["buf2"]), p


# ---- the instantiation matrix on two devices (tests/kernel_matrix.py): chunked kinds, chunked fused t0, the kernel chain -----
import kernel_matrix as km  # noqa: E402
from gpu_helpers import run_matrix_case  # noqa: E402

MATRIX_2 = km.two_device_cases()


@pytest.mark.parametrize("case", MATRIX_2, ids=[c.id for c in MATRIX_2])
def test_kernel_matrix_two_devices(case, monkeypatch):
    """Two-device cases of the matrix (odd lengths split unevenly): forward and backward per device against numpy's fftn in
    complex128, max|err| / rms(ref) <= 1e-13 log2 N (fp64) / 1e-6 log2 N (fp32), the scaled round trip, and the plan's path
    (fused, kernel chain, exchange)."""
    need(case.P)
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    run_matrix_case(case)


def test_kernel_matrix_error_report():
    """prints the worst error / bound per precision of the matrix cases that ran in this session (no assertion)"""
    print("\nkernel matrix:", km.report() or "no case ran")
