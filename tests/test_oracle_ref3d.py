"""Pins the oracle -- stage by stage -- on the reference's OWN HOT-PATH CODE, executed.

oracle/ref_3dmpifft compiles 3dmpifft_opt/include/fft_mpi_3d_api.cpp (plan creation, TransInfo tables, fftZY,
localTransposeUneven, slabAlltoall, fftX, fft_mpi_execute_dft_3d_c2c), kernel_func.cpp (the pack / unpack kernels),
fast_transpose/kernels_{201,120}.cpp (the cuTranspose tile kernels) and the FFT engine templateFFT/src/templateFFT.cpp (the
kernel generator) from the reference sources, in place, against a HIP-on-CPU shim and runs them on host memory: GPU threads
are fibers, and the kernels the engine generates at run time are compiled with g++ in place of hiprtc -- so the butterflies
and twiddles that run are the reference's too.  What that code produced is committed:

* tests/golden/ref3d_vectors.json (made by tests/golden/make_ref3d_vectors.py): BOTH plan buffers of every device after EVERY
  stage, the outputs and the exchange tables -- compared with both restatements (oracle_fft.c and the numpy twin) and, for
  the tables / counts / device policy, with the product library's host logic (libdfft.so; no GPU needed for those entry points);
* tests/golden/ref_samples.npz (made by tests/golden/make_ref_samples.py): random inputs over even and uneven splits up to 8
  devices, both directions, the engine's lines and radix schedules, BASELINE config 1 -- outputs too large to commit stored as a
  fixed sample (oracle.sampled) -- against numpy's fftn, against the oracle stage by stage, and against the product's recorded
  multi-device schedule interpreted on the CPU (tests/test_dry_run.py).

Only test_live_both_engines_agree_on_the_whole_path runs the reference itself (oracle/_ref) and skips without it."""
import json
import os

import numpy as np
import pytest

import distributedfft_b200 as dfft
from oracle import BACKWARD, FORWARD, COracle, NumpySlab, SlabGeometry, build_ref3d, proper_device_num, sampled

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 2e-13          # absolute, on O(1) inputs of <= 10^4 points: DFT vs Stockham vs pocketfft rounding


@pytest.fixture(scope="module")
def co():
    return COracle()


@pytest.fixture(scope="module")
def gold():
    with open(os.path.join(HERE, "golden", "ref3d_vectors.json")) as f:
        return json.load(f)


def c(v):
    a = np.asarray(v, dtype=np.float64)
    return a[:, 0] + 1j * a[:, 1]


def test_both_restatements_match_the_executed_reference_at_every_stage_boundary(co, gold):
    assert "fft_mpi_3d_api.cpp" in gold["library"] and "kernel_func.cpp" in gold["library"] and "templateFFT.cpp" in gold["library"]
    assert gold["engine"] == "templatefft"        # the vectors come from the reference's own generated FFT kernels
    for case in gold["cases"]:
        n0, n1, n2 = case["shape"]
        P, direction = case["devices"], case["direction"]
        g = SlabGeometry(n0, n1, n2, P)
        ns = NumpySlab(n0, n1, n2, P)
        ins = [c(b) for b in case["inputs"]]
        assert [b.size for b in ins] == [g.max_count(p) for p in range(P)]
        for s in range(4):
            for twin in (False, True):
                b1 = [b.copy() for b in ins]
                b2 = [np.zeros_like(b) for b in ins]
                if twin:
                    ns.execute(b1, b2, direction, stop_after=s)
                else:
                    co.slab_execute(g, b1, b2, direction, stop_after=s)
                for p in range(P):
                    st = case["stages"][p][s]
                    assert np.abs(b1[p] - c(st["buffer1"])).max() <= TOL, (case["shape"], P, direction, "stage", s, "bufferDev1", p, twin)
                    if not twin:      # (the numpy twin only keeps the buffer a stage produces; oracle_fft.c mirrors both)
                        assert np.abs(b2[p] - c(st["buffer2"])).max() <= TOL, (case["shape"], P, direction, "stage", s, "bufferDev2", p)
                    else:
                        live = b2[p] != 0
                        assert np.abs(b2[p][live] - c(st["buffer2"])[live]).max(initial=0) <= TOL
        # the result the caller sees
        b1 = [b.copy() for b in ins]
        b2 = [np.zeros_like(b) for b in ins]
        co.slab_execute(g, b1, b2, direction)
        for p in range(P):
            assert np.abs(b2[p] - c(case["outputs"][p])).max() <= TOL
        # ... and it IS the 3-D transform (forward: y-slabs [y_l][z][x]; backward: x-slabs [x_l][y][z], unnormalised)
        if direction == FORWARD:
            A = np.concatenate([ins[p][: g.in_count(p)] for p in range(P)]).reshape(n0, n1, n2)
            F = np.fft.fftn(A)
            for q in range(P):
                ref = F[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1)
                assert np.abs(c(case["outputs"][q])[: ref.size] - ref).max() <= TOL * 10


def test_binary_fixture_of_the_gpu_test_matches_the_oracle(co):
    """tests/golden/ref3d_case_8x16x32.npz (what tests/test_gpu_zz_reference_golden.py holds the CUDA path against): the
    oracle reproduces the executed reference's forward and backward outputs."""
    z = np.load(os.path.join(HERE, "golden", "ref3d_case_8x16x32.npz"))
    n0, n1, n2 = (int(v) for v in z["shape"])
    g = SlabGeometry(n0, n1, n2, 1)
    for src, want, direction in ((z["input"], z["forward"], FORWARD), (z["forward"], z["backward"], BACKWARD)):
        b1 = [src.copy()]
        b2 = [np.zeros_like(src)]
        co.slab_execute(g, b1, b2, direction)
        assert np.abs(b2[0] - want).max() <= 1e-13 * np.log2(src.size) * np.abs(want).max()
    assert np.abs(z["forward"] - np.fft.fftn(z["input"].reshape(n0, n1, n2)).transpose(1, 2, 0).reshape(-1)).max() <= 1e-12
    assert np.abs(z["backward"] / z["input"].size - z["input"]).max() <= 1e-13


def test_exchange_tables_counts_and_device_policy_match_the_executed_reference(co, gold, n_gpus):
    """Integers, so exact: the oracle's AND the product library's TransInfo tables (dfft_exchange_table), getMaxDataCount
    (dfft_max_data_count) and the device-count policy (dfft_init) against what the reference's own functions returned (with
    more devices than any row wants; dfft_init, like the reference, uses at most the GPUs present)."""
    for case in gold["cases"] + gold["table_cases"]:
        n0, n1, n2 = case["shape"]
        P, direction = case["devices"], case["direction"]
        t = np.asarray(case["tables"])
        for p in range(P):
            mine = dfft.exchange_table(n0, n1, n2, P, p, direction)
            orc = co.exchange_table(n0, n1, n2, P, p, direction)
            for j, k in enumerate(("scount", "soffset", "rcount", "roffset")):
                assert list(mine[k]) == list(t[p, :, j]) == list(orc[k]), (case["shape"], P, direction, p, k)
        if "max_data_count" in case:
            for last in (False, True):
                assert dfft.getMaxDataCount(n0, n1, n2, P, last) == case["max_data_count"][int(last)] == co.lib.oracle_max_data_count(n0, n1, n2, P, int(last))
    for row in gold["device_policy"]:
        assert proper_device_num(row["n0"], row["wanted"]) == row["proper"]
        usable = min(row["wanted"], n_gpus) if n_gpus else row["wanted"]
        want = row["proper"] if usable == row["wanted"] else proper_device_num(row["n0"], usable)
        assert dfft.fft_mpi_init([row["n0"], 64, 4], row["wanted"])[0] == want


@pytest.fixture(scope="module")
def rec():
    return np.load(os.path.join(HERE, "golden", "ref_samples.npz"))


@pytest.fixture(scope="module")
def ref():
    if build_ref3d() is None:
        pytest.skip("oracle/_ref/libref3dmpifft.so not built and the reference sources are absent")
    from oracle import Ref3dmpifft
    return Ref3dmpifft()


def _inputs(g, A, direction):
    if direction == FORWARD:
        return NumpySlab(g.n0, g.n1, g.n2, g.P).scatter_input(A)
    ins = []
    for q in range(g.P):
        b = np.zeros(g.max_count(q), dtype=np.complex128)
        blk = A[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1)
        b[: blk.size] = blk
        ins.append(b)
    return ins


def _cat(bufs, counts=None):
    """the per-device buffers one after the other (the recorded samples are taken of this)"""
    return np.concatenate(bufs if counts is None else [b[:n] for b, n in zip(bufs, counts)])


def _close(full, recorded, tol):
    """the recorded sample of a reference output against the same positions of `full`"""
    return np.abs(sampled(full, recorded.size) - recorded).max() <= tol


LIVE = [(1, 8, 8, 8), (2, 8, 8, 8), (3, 10, 9, 4), (3, 9, 10, 4), (4, 12, 10, 8), (4, 16, 8, 8), (8, 16, 16, 16), (3, 15, 22, 26), (5, 14, 9, 6), (8, 24, 16, 16), (7, 20, 27, 4)]


@pytest.mark.parametrize("P,n0,n1,n2", LIVE)
def test_live_executed_reference_vs_numpy_oracle_and_the_products_schedule(co, rec, P, n0, n1, n2):
    from test_dry_run import simulate
    g = SlabGeometry(n0, n1, n2, P)
    rng = np.random.default_rng(n0 * 1000 + n1 * 10 + P)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    key = f"exec/{P}x{n0}x{n1}x{n2}"
    assert np.array_equal(A.reshape(-1)[:4], rec[key + "/input_head"]), "the recorded input is not the one regenerated here"
    for direction in (FORWARD, BACKWARD):
        d = f"{key}/{direction}"
        ins = _inputs(g, A, direction)
        outs = rec[d + "/out"]       # the stage-by-stage run; the reference's fft_mpi_execute_dft_3d_c2c gave the same when recorded
        tol = 1e-13 * np.log2(A.size) * np.abs(np.fft.fftn(A)).max()
        # (1) numpy: forward = fftn in y-slabs; backward = unnormalised ifftn in x-slabs
        if direction == FORWARD:
            F = np.fft.fftn(A)
            want = [F[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1) for q in range(P)]
        else:
            B = np.fft.ifftn(A) * A.size
            want = [B[p * g.xd: p * g.xd + g.n0l(p)].reshape(-1) for p in range(P)]
        counts = [w.size for w in want]
        assert _close(_cat(want), outs, tol)
        # (2) the oracle, both buffers at every stage boundary
        stages = rec[d + "/stages"]
        for s in range(4):
            b1 = [b.copy() for b in ins]
            b2 = [np.zeros_like(b) for b in ins]
            co.slab_execute(g, b1, b2, direction, stop_after=s)
            assert _close(_cat(b1), stages[s, 0], tol), (s, "bufferDev1")
            assert _close(_cat(b2), stages[s, 1], tol), (s, "bufferDev2")
        # (3) the product's recorded schedule (P2P fused, P2P two-sweep, NCCL), interpreted on the CPU
        for flags in (dfft.EXCHANGE_P2P, dfft.EXCHANGE_P2P | dfft.NO_FUSE, dfft.EXCHANGE_NCCL):
            got, _, _ = simulate(n0, n1, n2, P, direction, ins, flags)
            assert _close(_cat(got, counts), outs, tol), flags
        # (4) tables
        tables = rec[d + "/tables"]
        for p in range(P):
            mine = dfft.exchange_table(n0, n1, n2, P, p, direction)
            for j, k in enumerate(("scount", "soffset", "rcount", "roffset")):
                assert list(mine[k]) == list(tables[p, :, j])


def test_live_counts_and_policy_sweep(rec):
    rows = rec["counts/max_data_count"]
    assert len(rows) > 100
    for P, n0, n1, n2, last, want in rows.tolist():
        assert dfft.getMaxDataCount(n0, n1, n2, P, last) == want
    policy = rec["counts/proper_device_num"]
    for n0 in range(1, 70):
        for w in range(1, 9):
            assert proper_device_num(n0, w) == policy[n0 - 1, w - 1], (n0, w)


def test_oracle_engine_matches_the_references_generated_fft_kernels(co, gold):
    """The 1-D / 2-D engine alone, on the baseline's axis lengths (512, 768, 1024 among them): oracle_fft.c's Stockham engine and
    numpy against what the reference's generated kernels produced (committed vectors)."""
    for case in gold["engine_cases"]:
        x = c(case["input"]).reshape(case["shape"])
        n = x.size
        tol = 1e-15 * 8 * np.log2(n) * np.abs(c(case["forward"])).max()
        if case["fftdim"] == 1:
            mine = co.fft_axis(x.reshape(1, -1), 1, -1).reshape(-1)
            npy = np.fft.fft(x)
        else:
            mine = co.fft_axis(co.fft_axis(x, 1, -1), 0, -1).reshape(-1)
            npy = np.fft.fft2(x).reshape(-1)
        assert np.abs(mine - c(case["forward"])).max() <= tol, case["shape"]
        assert np.abs(npy.reshape(-1) - c(case["forward"])).max() <= tol, case["shape"]
        if "backward" in case:
            if case["fftdim"] == 1:
                mine = co.fft_axis(x.reshape(1, -1), 1, +1).reshape(-1)
            else:
                mine = co.fft_axis(co.fft_axis(x, 1, +1), 0, +1).reshape(-1)
            assert np.abs(mine - c(case["backward"])).max() <= tol, case["shape"]      # unnormalised inverse (templateFFT.cpp:5946 normalize = 0)


ENGINE_LENGTHS = [2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 15, 16, 18, 20, 21, 24, 25, 27, 28, 30, 32, 35, 36, 48, 49, 64, 81, 96, 100, 125, 128, 243, 256, 343,
                  512, 625, 768, 1000, 1024, 2048, 4096, 8192]
ENGINE_REJECTED = (11, 13, 17, 22, 26, 33)


def test_live_reference_engine_lengths_vs_oracle_numpy_and_the_products_length_policy(co, rec):
    """Every length the reference's generator takes up to 4096 in a sample, plus 8192 (its multi-upload path): the generated
    kernels vs numpy and vs oracle_fft.c; the product library supports (dfft_length_kind != 0) every such length up to its
    single-line limit -- it is a superset (radix 11 and 13 are extra)."""
    rng = np.random.default_rng(11)
    for n in ENGINE_LENGTHS:
        a = rng.standard_normal((2, n)) + 1j * rng.standard_normal((2, n))
        if n == ENGINE_LENGTHS[0]:
            assert np.array_equal(a.reshape(-1)[:4], rec["engine/input_head"])
        got, back = rec[f"engine/{n}/forward,backward"]
        want = np.fft.fft(a, axis=1)
        tol = 1e-15 * 8 * np.log2(n) * np.abs(want).max()
        assert _close(want, got, tol), n
        if n <= 4096:
            assert _close(co.fft_axis(a, 1, -1), got, tol), n
            assert dfft.length_kind(n) != 0, n
        assert np.abs(back / n - sampled(a, back.size)).max() <= 1e-13
    assert rec["engine/rejected"].all()            # the reference's generator has no radix above 8; the product adds 11 and 13
    assert dfft.length_kind(11) != 0 and dfft.length_kind(26) != 0 and dfft.length_kind(17) == 0
    # a 2-D plane (the fftZY configuration: size = {N2, N1}, fft_mpi_3d_api.cpp:381-384)
    a = rng.standard_normal((3, 12, 16)) + 1j * rng.standard_normal((3, 12, 16))
    assert np.array_equal(a.reshape(-1)[:4], rec["engine/plane/input_head"])
    assert _close(np.fft.fft2(a), rec["engine/plane/forward"], 1e-13)


def test_live_both_engines_agree_on_the_whole_path(ref):
    """The DFT stand-in (used only for sizes with a prime factor above 7, which the reference's generator cannot do) and the
    reference's generated kernels give the same slabs."""
    if ref.set_engine("templatefft") != "templatefft":
        pytest.skip("libtemplatefft_cpu.so not built")
    rng = np.random.default_rng(12)
    for (P, n0, n1, n2) in [(2, 8, 8, 8), (3, 10, 9, 4), (4, 12, 10, 8)]:
        g = SlabGeometry(n0, n1, n2, P)
        A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
        for direction in (FORWARD, BACKWARD):
            ins = _inputs(g, A, direction)
            assert ref.set_engine("templatefft") == "templatefft" and ref.engine_used(n0, n1, n2) == "templatefft"
            a, _, _ = ref.execute(g, ins, direction)
            assert ref.set_engine("dft") == "dft"
            b, _, _ = ref.execute(g, ins, direction)
            ref.set_engine("templatefft")
            for p in range(P):
                assert 0 < np.abs(a[p] - b[p]).max() <= 1e-12       # different arithmetic, same transform


@pytest.mark.parametrize("P", [1, 4])
def test_live_baseline_config_c1_on_the_executed_reference(co, rec, P):
    """BASELINE.json configs[0]: 64x64x64 C2C forward + inverse with the round-trip max-error check of the reference driver
    (fftSpeed3d_c2c.cpp:79-91: |x - ifft(fft(x)) / N^3| <= 1e-11) -- run on the reference's own code (its generated FFT kernels
    included), and the forward spectrum compared with the oracle's and numpy's."""
    n = 64
    g = SlabGeometry(n, n, n, P)
    a = np.zeros(n * n * n, dtype=np.complex128)
    co.fill_minstd(a, 4242)
    A = a.reshape(n, n, n)
    ins = NumpySlab(n, n, n, P).scatter_input(A)
    spec, back = rec[f"c1/{P}/forward,backward"]
    b1 = [b.copy() for b in ins]
    b2 = [np.zeros_like(b) for b in ins]
    co.slab_execute(g, b1, b2, FORWARD)
    F = np.fft.fftn(A)
    want = [F[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1) for q in range(P)]
    tol = 1e-12 * 18 * np.abs(F).max()
    assert _close(_cat(want), spec, tol)
    assert _close(_cat(b2, [w.size for w in want]), spec, tol)
    assert np.abs(back / n ** 3 - sampled(_cat(ins, [g.in_count(p) for p in range(P)]), back.size)).max() <= 1e-11


RADIX_POW = (2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 3, 9, 27, 81, 243, 2187, 5, 25, 125, 625, 3125, 7, 49, 343)
RADIX_MIXED = (6, 12, 20, 24, 48, 96, 100, 360, 768, 1000, 3000)
RADIX_MULTI = (6144, 6400, 8192)
RADIX_REJECTED = (22, 13)


def test_live_radix_schedules_of_the_references_generator(co, rec):
    """What the reference's FFTScheduler actually picks (read back from the plans the executed generator built) against the
    radix policy restated in oracle_fft.c / used by the product's run-time-scheduled kernel (templateFFT.cpp:3956-3963,
    4540-4550, 4580-4588): identical for powers of 2, 3, 5 and 7 -- 512 = 8.8.8, 1024 = 8.8.8.2, 4096 = 8.8.8.8 among them --;
    for mixed lengths the generator merges the 2s into 8s / 4s only when the register count of the other radix allows it
    (:4540-4550: 768 = 4.4.4.4.3 there, 8.8.4.3 here), a choice that changes rounding, not the transform (the values are
    compared in test_live_reference_engine_lengths_...).  Lengths beyond one shared-memory line use several uploads."""
    table = {int(r[0]): r[1:].tolist() for r in rec["radix"]}         # n, uploads (-1: not taken), radices..., 0-padded

    def schedule(n):
        r = table[n]
        return None if r[0] == -1 else ([x for x in r[1:] if x], r[0])
    for n in RADIX_POW:
        radices, uploads = schedule(n)
        assert uploads == 1 and radices == co.radix_schedule(n), (n, radices)
    for n in RADIX_MIXED:
        radices, uploads = schedule(n)
        assert uploads == 1 and int(np.prod(radices)) == n == int(np.prod(co.radix_schedule(n))) and set(radices) <= {2, 3, 4, 5, 7, 8}
    assert schedule(768)[0] == [4, 4, 4, 4, 3] and co.radix_schedule(768) == [8, 8, 4, 3]
    for n in RADIX_MULTI:            # multi-upload (four-step) lengths of the reference: two kernels
        radices, uploads = schedule(n)
        assert uploads == 2 and int(np.prod(radices)) == n
    assert all(schedule(n) is None for n in RADIX_REJECTED)


PIPELINED = [(4, 8, 12, 64, dfft.EXCHANGE_P2P), (2, 64, 64, 64, dfft.EXCHANGE_P2P), (3, 10, 9, 128, dfft.EXCHANGE_P2P), (4, 8, 8, 64, dfft.EXCHANGE_NCCL),
             (8, 16, 16, 64, dfft.EXCHANGE_P2P)]


@pytest.mark.parametrize("P,n0,n1,n2,flags", PIPELINED)
def test_live_pipelined_schedules_of_the_product_vs_the_executed_reference(rec, P, n0, n1, n2, flags):
    """The z-part pipelines (kernel chain for the cube, two streams otherwise, P2P and NCCL, forward and backward): the product's
    recorded schedule, interpreted on the CPU, gives the slabs the reference's executed code gives."""
    from test_dry_run import simulate
    g = SlabGeometry(n0, n1, n2, P)
    rng = np.random.default_rng(P * 100 + n2)
    A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
    key = f"pipelined/{P}x{n0}x{n1}x{n2}"
    assert np.array_equal(A.reshape(-1)[:4], rec[key + "/input_head"])
    scale = np.abs(np.fft.fftn(A)).max()
    for direction, outs in zip((FORWARD, BACKWARD), rec[key + "/forward,backward"]):
        ins = _inputs(g, A, direction)
        got, names, _ = simulate(n0, n1, n2, P, direction, ins, flags | dfft.FORCE_PIPELINE)
        assert len(names[0]) > 4, names[0]          # really cut into parts
        counts = [g.out_count(p) if direction == FORWARD else g.in_count(p) for p in range(P)]
        assert _close(_cat(got, counts), outs, 1e-13 * np.log2(A.size) * scale), direction
