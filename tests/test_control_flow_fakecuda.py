"""CPU test of the NON-dry host control flow of libdfft.so.

Round 1 shipped a library whose every real `dfft_execute` spun forever on the host (a self-recursive event
helper) while the CPU suite stayed green, because it only ever created DFFT_DRY_RUN plans.  Here the
library's own object files are linked against tests/fakecuda/fake_cudart.cpp (device memory = host memory,
launches = counted no-ops) and real plans are driven create -> execute -> timings -> destroy for one
device and for 2/4 device-threads of a local communicator, in every exchange mode that needs no NCCL,
under a hard timeout.  A hang, a crash or a bootstrap deadlock fails in seconds, without a GPU."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "distributedfft_b200")
FAKE_LIB = os.path.join(PKG, "build", "libdfft_fakecuda.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.fixture(scope="module")
def fake_lib():
    sys.path.insert(0, ROOT)
    from distributedfft_b200 import build as b
    b.build()
    objs = [os.path.join(PKG, "build", s.replace(".cu", ".o")) for s in b.LIB_SOURCES]
    stub_src = os.path.join(ROOT, "tests", "fakecuda", "fake_cudart.cpp")
    stub_obj = os.path.join(PKG, "build", "fake_cudart.o")
    newest = max(os.path.getmtime(p) for p in objs + [stub_src])
    if not os.path.exists(FAKE_LIB) or os.path.getmtime(FAKE_LIB) < newest:
        subprocess.run(["g++", "-O1", "-fPIC", "-std=c++17", "-c", stub_src, "-o", stub_obj], check=True)
        subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "none", "-o", FAKE_LIB] + objs +
                       [stub_obj, "-ldl", "-lpthread", "-ccbin", "/usr/bin/g++"], check=True)
    return FAKE_LIB


WORKER = textwrap.dedent(r'''
    import ctypes, sys, threading
    sys.path.insert(0, sys.argv[1])
    import distributedfft_b200.api as api
    api.LIB_PATH = sys.argv[2]          # the fake-runtime build of the same objects
    api._lib = None
    import distributedfft_b200 as dfft
    L = dfft.lib()
    L.fakecuda_launches.restype = ctypes.c_longlong
    L.fakecuda_event_records.restype = ctypes.c_longlong
    L.fakecuda_live_allocations.restype = ctypes.c_longlong

    def drive(n0, n1, n2, P, flags, precision=dfft.DOUBLE, executes=3):
        comm = dfft.LocalComm(P) if P > 1 else None
        errs, launches = [], [0] * P
        def worker(p):
            try:
                for direction in (dfft.FORWARD, dfft.BACKWARD):
                    mc = dfft.getMaxDataCount(n0, n1, n2, P, p == P - 1)
                    a = dfft.fft_mpi_alloc_local_memory(mc, dfft.ALLOC_DEV, precision)
                    b = dfft.fft_mpi_alloc_local_memory(mc, dfft.ALLOC_DEV, precision)
                    plan = dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, a, b, comm, p, P, direction, precision, flags)
                    for _ in range(executes):
                        plan.execute()
                    plan.synchronize()
                    t = plan.timings(); pt = plan.pass_timings()
                    assert len(t) == 5 and t[4] > 0 and len(pt) == 3
                    launches[p] += plan.launches
                    assert plan.launches >= 2
                    plan.destroy()
                    L.dfft_free_local(a, dfft.ALLOC_DEV); L.dfft_free_local(b, dfft.ALLOC_DEV)
            except Exception:
                import traceback
                errs.append(traceback.format_exc())
        if P == 1:
            worker(0)
        else:
            th = [threading.Thread(target=worker, args=(p,)) for p in range(P)]
            [t.start() for t in th]; [t.join() for t in th]
        if comm: comm.destroy()
        assert not errs, "\n".join(errs)
        return launches

    before = L.fakecuda_launches()
    for flags in (0, dfft.FORCE_FUSE, dfft.NO_FUSE, dfft.EXCHANGE_STAGED, dfft.SCALE_BACKWARD, dfft.NATURAL_SPECTRUM):
        drive(64, 64, 64, 1, flags)
        drive(12, 10, 24, 1, flags, dfft.FLOAT)
    for P in (2, 4):
        for flags in (dfft.EXCHANGE_P2P, dfft.EXCHANGE_P2P | dfft.NO_FUSE, dfft.EXCHANGE_P2P | dfft.OVERLAP_X, dfft.EXCHANGE_STAGED):
            drive(64, 64, 64, P, flags)
            drive(12, 10, 24, P, flags)          # uneven split (short last slab), generic lengths
        drive(8, 128, 128, P, dfft.EXCHANGE_P2P | dfft.FORCE_PIPELINE)     # stream-pipelined (4 z-parts, two streams), fused part 0
        drive(8, 12, 128, P, dfft.EXCHANGE_P2P | dfft.FORCE_PIPELINE)      # ... two-sweep t0
        drive(8, 128, 128, P, dfft.EXCHANGE_P2P | dfft.NO_PIPELINE)
        drive(128, 128, 128, P, dfft.EXCHANGE_P2P | dfft.FORCE_PIPELINE, executes=2)   # cube: the kernel chain [Z+Y0][Y1+X0]..[X last] forward
    # 8 device-threads (the reference's largest node): plain, two-sweep, kernel chain, uneven split
    for flags in (dfft.EXCHANGE_P2P, dfft.EXCHANGE_P2P | dfft.NO_FUSE, dfft.EXCHANGE_STAGED):
        drive(64, 64, 64, 8, flags, executes=2)
    drive(128, 128, 128, 8, dfft.EXCHANGE_P2P | dfft.FORCE_PIPELINE, executes=2)
    drive(30, 22, 24, 8, dfft.EXCHANGE_P2P, executes=2)
    # the host-buffer entry points and the lines engine
    cnt = 16 * 16 * 16
    buf = dfft.fft_mpi_alloc_local_memory(cnt, dfft.ALLOC_DEV)
    plan = dfft.fft_mpi_plan_dft_c2c_3d(16, 16, 16, buf, None, None, 0, 1, dfft.FORWARD)
    hin = dfft.fft_mpi_alloc_local_memory(cnt, dfft.ALLOC_CPU); hout = dfft.fft_mpi_alloc_local_memory(cnt, dfft.ALLOC_CPU)
    plan.execute_host(hin, hout); plan.execute_host_async(hin, hout); plan.synchronize(); plan.destroy()
    for p_ in (buf,): L.dfft_free_local(p_, dfft.ALLOC_DEV)
    for p_ in (hin, hout): L.dfft_free_local(p_, dfft.ALLOC_CPU)
    # what bench.py's e2e leg does at N > 1: TWO collective plans per device, driven alternately through the host-buffer entry
    # points (step i's D2H overlaps step i+1's H2D) -- 2 and 8 device-threads
    def two_plans_in_flight(P, n):
        comm = dfft.LocalComm(P)
        errs = []
        def worker(p):
            try:
                mc = dfft.getMaxDataCount(n, n, n, P, p == P - 1)
                bufs = [dfft.fft_mpi_alloc_local_memory(mc, dfft.ALLOC_DEV) for _ in range(4)]
                host = [dfft.fft_mpi_alloc_local_memory(mc, dfft.ALLOC_CPU) for _ in range(4)]
                plans = [dfft.fft_mpi_plan_dft_c2c_3d(n, n, n, bufs[2 * k], bufs[2 * k + 1], comm, p, P, dfft.FORWARD, dfft.DOUBLE, dfft.EXCHANGE_P2P) for k in range(2)]
                for step in range(6):
                    k = step % 2
                    if step >= 2:
                        plans[k].synchronize()
                    plans[k].execute_host_async(host[2 * k], host[2 * k + 1])
                for pl in plans:
                    pl.synchronize()
                for pl in plans:
                    pl.destroy()
                for b in bufs: L.dfft_free_local(b, dfft.ALLOC_DEV)
                for b in host: L.dfft_free_local(b, dfft.ALLOC_CPU)
            except Exception:
                import traceback
                errs.append(traceback.format_exc())
        th = [threading.Thread(target=worker, args=(p,)) for p in range(P)]
        [t.start() for t in th]; [t.join() for t in th]
        comm.destroy()
        assert not errs, "\n".join(errs)
    two_plans_in_flight(2, 64)
    two_plans_in_flight(8, 64)
    data = dfft.fft_mpi_alloc_local_memory(4096 * 4, dfft.ALLOC_DEV)
    dfft.fft_lines(data, 4096, 1, 4, 4, 4096, 4 * 4096, dfft.FORWARD)
    lp = dfft.LinesPlan(two_d=(64, 32, 2)); lp.execute(data, dfft.FORWARD); lp.execute(data, dfft.BACKWARD); lp.synchronize(); lp.destroy()
    L.dfft_free_local(data, dfft.ALLOC_DEV)
    # errors still come back as status codes on the real path
    try:
        dfft.fft_mpi_plan_dft_c2c_3d(17, 16, 16, 1, 2, None, 0, 1, dfft.FORWARD)
        raise SystemExit("unsupported length accepted")
    except dfft.DfftError:
        pass
    # one participant of a collective plan creation fails (null input pointer): its peer must get an error back, not hang
    comm = dfft.LocalComm(2)
    out = {}
    def half(p_):
        a = dfft.fft_mpi_alloc_local_memory(16 * 16 * 16, dfft.ALLOC_DEV)
        try:
            pl = dfft.fft_mpi_plan_dft_c2c_3d(16, 16, 16, a if p_ == 0 else None, None, comm, p_, 2, dfft.FORWARD, dfft.DOUBLE, dfft.EXCHANGE_P2P)
            pl.destroy(); out[p_] = "created"
        except dfft.DfftError as e:
            out[p_] = "error"
        L.dfft_free_local(a, dfft.ALLOC_DEV)
    th = [threading.Thread(target=half, args=(k,)) for k in range(2)]
    [t.start() for t in th]; [t.join(30) for t in th]
    assert out == {0: "error", 1: "error"}, out
    comm.destroy()
    assert L.fakecuda_launches() - before > 100 and L.fakecuda_event_records() > 100
    assert L.fakecuda_live_allocations() == 0, ("leak", L.fakecuda_live_allocations())
    print("fakecuda control flow ok: %d launches, %d event records" % (L.fakecuda_launches(), L.fakecuda_event_records()))
''')


def test_non_dry_plans_run_to_completion_on_a_fake_runtime(fake_lib, tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, DFFT_VERBOSE="1")
    r = subprocess.run([sys.executable, str(script), ROOT, fake_lib], capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "fakecuda control flow ok" in r.stdout


DRIVER_SRC = os.path.join(PKG, "driver", "distFFT.cpp")


@pytest.mark.parametrize("P", [1, 2, 8])
def test_reference_driver_through_the_cxx_shim_on_a_fake_runtime(fake_lib, tmp_path, P):
    """The reference-facing C++ surface (include/fft_mpi_3d_api.h: fft_mpi_init, getMaxDataCount, fft_mpi_alloc_local_memory,
    fft_mpi_plan_dft_c2c_3d, fft_mpi_execute_dft_3d_c2c, fft_mpi_destroy_plan -- api.h:68-74) driven by driver/distFFT.cpp (the
    call sequence of fftSpeed3d_c2c.cpp:42-138, one host thread per device like its OpenMP region) against the fake-runtime
    build: the whole program runs to its report block without a GPU.  Numbers are meaningless here (kernels are no-ops);
    the control flow, the printed surface and the exit code are what is checked."""
    exe = tmp_path / "distFFT_fake"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", DRIVER_SRC, "-o", str(exe),
                    fake_lib, "-Wl,-rpath," + os.path.dirname(fake_lib), "-lpthread"], check=True)
    env = dict(os.environ, FAKECUDA_DEVICES="8")
    r = subprocess.run([str(exe), "32", "32", "32", str(P)], capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = r.stdout
    assert "allocate %d devices to node 0" % P in out                     # api.cpp:270
    assert out.count("data count in device") == P                          # api.cpp:285
    assert out.count("t0: ") >= 4 * P                                      # one stage line per forward execute and device (api.cpp:201)
    for key in ("distributed FFT performance test", "Size:             32x32x32", "MPI ranks:        %d" % P, "Forward FFT time:", "Performance:",
                "Max error:"):                                             # drv.cpp:126-138
        assert key in out, key
    # the reference's argument check (drv.cpp:33-36)
    r = subprocess.run([str(exe), "32", "32"], capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode != 0 and "The format of arguments should be [NX, NY, NZ, GPU_COUNT]!" in r.stdout


def test_driver_stdout_surface_is_the_reference_drivers(fake_lib, tmp_path):
    """The reference's OWN driver program (3dmpifft_opt/fftSpeed3d_c2c.cpp compiled in place against the HIP-on-CPU shim, one
    device; its stdout is recorded in tests/golden/distFFT_ref_stdout.json by tests/golden/make_ref_samples.py) and this repo's
    driver/distFFT.cpp (against the fake CUDA runtime) are run with the same arguments: with every number replaced by '#', the
    reference's stdout must be, line for line and in order, a subsequence of ours (ours adds lines after the report block)."""
    import json
    import re
    with open(os.path.join(ROOT, "tests", "golden", "distFFT_ref_stdout.json")) as f:
        theirs = json.load(f)
    exe = tmp_path / "distFFT_fake"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", DRIVER_SRC, "-o", str(exe),
                    fake_lib, "-Wl,-rpath," + os.path.dirname(fake_lib), "-lpthread"], check=True)
    ours = subprocess.run([str(exe)] + theirs["args"], capture_output=True, text=True, timeout=60, env=dict(os.environ, FAKECUDA_DEVICES="8"))
    assert ours.returncode == 0 and theirs["returncode"] == 0, ours.stderr

    def shape(text):
        out = []
        for line in text.splitlines():
            line = re.sub(r"on \S+ ready", "on HOST ready", line)
            line = re.sub(r"[-+]?(\d+\.?\d*|\.\d+)([eE][-+]?\d+)?|inf|nan", "#", line)
            line = re.sub(r"\s+", " ", line).strip()
            if line:
                out.append(line)
        return out
    a, b = shape(theirs["stdout"]), shape(ours.stdout)
    assert "Size: #x#x#" in a and "Max error: #" in a and a.count("t#: #, t#: #, t#: #, t#: #, total: #") == 4
    it = iter(b)
    missing = [line for line in a if line not in it]          # `in` consumes the iterator: an ordered-subsequence check
    assert not missing, (missing, b)
    # the reference's argument check (fftSpeed3d_c2c.cpp:28-31)
    ours_bad = subprocess.run([str(exe)] + theirs["bad_args"], capture_output=True, text=True, timeout=60)
    assert theirs["bad_args_returncode"] != 0 and ours_bad.returncode != 0
    assert [l for l in theirs["bad_args_stdout"].splitlines() if "format of arguments" in l] == [l for l in ours_bad.stdout.splitlines() if "format of arguments" in l] != []
