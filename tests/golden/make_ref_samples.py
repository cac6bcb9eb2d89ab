#!/usr/bin/env python
"""Generates tests/golden/ref_samples.npz and tests/golden/distFFT_ref_stdout.json by RUNNING the reference's own code, built
into oracle/_ref by oracle/ref_heffte/Makefile and oracle/ref_3dmpifft/Makefile from the reference sources:

* heFFTe 2.1.0 (stock backend): forward and backward world transforms (tests/test_oracle_ref.py);
* 3dmpifft_opt's hot path and its FFT engine, executed on the CPU: per-device outputs, both plan buffers after every stage,
  exchange tables, count and device policies, the engine's lines and radix schedules (tests/test_oracle_ref3d.py);
* the reference's driver program fftSpeed3d_c2c.cpp: its stdout (tests/test_control_flow_fakecuda.py).

The inputs are the ones the tests regenerate (same seeds; the first values are stored so a changed random stream is caught).
Outputs too large to commit are stored as a fixed sample (oracle.sampled): the tests compare the same positions of their own
results.  Per device buffers are concatenated before sampling.

    python tests/golden/make_ref_samples.py      (needs the reference sources where oracle.build_ref() looks for them)
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import BACKWARD, FORWARD, COracle, HeffteRef, NumpySlab, Ref3dmpifft, SlabGeometry, build_ref, build_ref3d, minstd_uniform, sampled  # noqa: E402
from test_oracle_ref import HEFFTE_LIVE  # noqa: E402
from test_oracle_ref3d import ENGINE_LENGTHS, ENGINE_REJECTED, LIVE, PIPELINED, RADIX_MIXED, RADIX_MULTI, RADIX_POW, RADIX_REJECTED, _inputs  # noqa: E402

K_OUT, K_STAGE, K_LINE, K_BIG = 96, 16, 32, 256


def cat(bufs, counts=None):
    return np.concatenate(bufs if counts is None else [b[:n] for b, n in zip(bufs, counts)])


def heffte(out):
    ref = HeffteRef()
    out["heffte/version"] = np.array(ref.version())
    for i, (n0, n1, n2, P, alg) in enumerate(HEFFTE_LIVE):
        vals, _ = minstd_uniform(n0 * n1 * n2, 4242) if n0 * n1 * n2 <= 8192 else (np.random.default_rng(3).random(n0 * n1 * n2), 0)
        A = (vals + 1j * np.roll(vals, 7)).reshape(n0, n1, n2)
        S = ref.fft3d(A, P, FORWARD, alg)
        B = ref.fft3d(S, P, BACKWARD, alg)
        out[f"heffte/{i}/input_head"] = A.reshape(-1)[:4]
        out[f"heffte/{i}/forward,backward"] = np.stack([sampled(S, 128), sampled(B, 128)])
    rng = np.random.default_rng(5)
    A = (rng.random((16, 12, 8)) + 1j * rng.random((16, 12, 8))).astype(np.complex64)
    out["heffte/float/input_head"] = A.reshape(-1)[:4]
    out["heffte/float/forward"] = sampled(ref.fft3d(A, 2, FORWARD), 512)


def ref3d(out):
    ref = Ref3dmpifft()
    assert ref.set_engine("templatefft") == "templatefft", "the samples must come from the reference's own FFT kernels"
    for (P, n0, n1, n2) in LIVE:
        g = SlabGeometry(n0, n1, n2, P)
        rng = np.random.default_rng(n0 * 1000 + n1 * 10 + P)
        A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
        key = f"exec/{P}x{n0}x{n1}x{n2}"
        out[key + "/input_head"] = A.reshape(-1)[:4]
        for direction in (FORWARD, BACKWARD):
            d = f"{key}/{direction}"
            ins = _inputs(g, A, direction)
            outs, tables, dumps = ref.execute(g, ins, direction, stages=True)
            whole, _, _ = ref.execute(g, ins, direction)          # the reference's own fft_mpi_execute_dft_3d_c2c
            assert all(np.array_equal(a, b) for a, b in zip(outs, whole))
            counts = [g.out_count(p) if direction == FORWARD else g.in_count(p) for p in range(P)]
            out[d + "/out"] = sampled(cat(outs, counts), K_OUT)
            out[d + "/stages"] = np.array([[sampled(cat([dumps[p][s][w] for p in range(P)]), K_STAGE) for w in range(2)] for s in range(4)])
            out[d + "/tables"] = tables
    rng = np.random.default_rng(5)
    rows = []
    for _ in range(200):
        P = int(rng.integers(1, 9))
        n0, n1, n2 = (int(rng.integers(1, 200)) for _ in range(3))
        if (P - 1) * -(-n0 // P) >= n0 or (P - 1) * -(-n1 // P) >= n1:
            continue
        for last in (0, 1):
            rows.append([P, n0, n1, n2, last, ref.max_data_count(n0, n1, n2, P, last)])
    out["counts/max_data_count"] = np.array(rows, dtype=np.int64)
    out["counts/proper_device_num"] = np.array([[ref.proper_device_num(n0, w) for w in range(1, 9)] for n0 in range(1, 70)], dtype=np.int64)
    # the FFT engine alone
    rng = np.random.default_rng(11)
    for n in ENGINE_LENGTHS:
        a = rng.standard_normal((2, n)) + 1j * rng.standard_normal((2, n))
        if n == ENGINE_LENGTHS[0]:
            out["engine/input_head"] = a.reshape(-1)[:4]
        got = ref.engine_fft(a)
        out[f"engine/{n}/forward,backward"] = np.stack([sampled(got, K_LINE), sampled(ref.engine_fft(got, inverse=True), K_LINE)])
    out["engine/rejected"] = np.array([ref.engine_fft(np.zeros(n, dtype=np.complex128)) is None for n in ENGINE_REJECTED])
    a = rng.standard_normal((3, 12, 16)) + 1j * rng.standard_normal((3, 12, 16))
    out["engine/plane/input_head"] = a.reshape(-1)[:4]
    out["engine/plane/forward"] = sampled(ref.engine_fft(a, 2), 64)
    rows = []                       # n, uploads (-1: length not taken), radices..., 0-padded
    for n in RADIX_POW + RADIX_MIXED + RADIX_MULTI + RADIX_REJECTED:
        s = ref.engine_schedule(n)
        rows.append([n, -1] if s is None else [n, s[1]] + s[0])
    out["radix"] = np.array([r + [0] * (16 - len(r)) for r in rows], dtype=np.int64)
    # BASELINE.json configs[0] on the executed reference
    n = 64
    a = np.zeros(n * n * n, dtype=np.complex128)
    COracle().fill_minstd(a, 4242)
    for P in (1, 4):
        g = SlabGeometry(n, n, n, P)
        ins = NumpySlab(n, n, n, P).scatter_input(a.reshape(n, n, n))
        spec, _, _ = ref.execute(g, ins, FORWARD)
        back, _, _ = ref.execute(g, spec, BACKWARD)
        out[f"c1/{P}/forward,backward"] = np.stack([sampled(cat(spec, [g.out_count(q) for q in range(P)]), K_BIG),
                                                    sampled(cat(back, [g.in_count(p) for p in range(P)]), K_BIG)])
    # the pipelined schedules' geometries
    for (P, n0, n1, n2, _flags) in PIPELINED:
        g = SlabGeometry(n0, n1, n2, P)
        rng = np.random.default_rng(P * 100 + n2)
        A = rng.standard_normal((n0, n1, n2)) + 1j * rng.standard_normal((n0, n1, n2))
        key = f"pipelined/{P}x{n0}x{n1}x{n2}"
        out[key + "/input_head"] = A.reshape(-1)[:4]
        res = []
        for direction in (FORWARD, BACKWARD):
            outs, _, _ = ref.execute(g, _inputs(g, A, direction), direction)
            res.append(sampled(cat(outs, [g.out_count(p) if direction == FORWARD else g.in_count(p) for p in range(P)]), 128))
        out[key + "/forward,backward"] = np.stack(res)


def driver_stdout():
    exe = os.path.join(ROOT, "oracle", "_ref", "distFFT_ref")
    good = subprocess.run([exe, "16", "16", "16", "1"], capture_output=True, text=True, timeout=120)
    bad = subprocess.run([exe, "16", "16"], capture_output=True, text=True, timeout=60)
    doc = {"generator": "tests/golden/make_ref_samples.py", "program": "3dmpifft_opt/fftSpeed3d_c2c.cpp of the reference, one device (oracle/_ref/distFFT_ref)",
           "args": ["16", "16", "16", "1"], "returncode": good.returncode, "stdout": good.stdout,
           "bad_args": ["16", "16"], "bad_args_returncode": bad.returncode, "bad_args_stdout": bad.stdout}
    with open(os.path.join(ROOT, "tests", "golden", "distFFT_ref_stdout.json"), "w") as f:
        json.dump(doc, f, indent=1)


def main():
    assert build_ref() and build_ref3d(), "the reference sources are needed to run the reference"
    out = {}
    heffte(out)
    ref3d(out)
    driver_stdout()
    path = os.path.join(ROOT, "tests", "golden", "ref_samples.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
