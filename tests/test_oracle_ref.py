"""Pins the restated oracle (oracle/oracle_fft.c + the numpy twin) on outputs of the EXECUTED reference: the
reference tree's own heFFTe 2.1.0 with its `stock` CPU backend (heffte/heffteBenchmark, the library the reference
benchmarks against), built by oracle/ref_heffte/Makefile into oracle/_ref/libheffte_ref.so.

* tests/golden/heffte_ref_vectors.json (made by tests/golden/make_heffte_ref_vectors.py): whole forward spectra;
* tests/golden/ref_samples.npz (made by tests/golden/make_ref_samples.py): forward and backward transforms of random and
  heFFTe-test inputs, even and uneven slab splits, every reshape algorithm, up to 64^3, stored as a fixed sample of each
  output (oracle.sampled).  Neither needs the reference sources or oracle/_ref."""
import json
import os

import numpy as np
import pytest

from oracle import BACKWARD, FORWARD, COracle, NumpySlab, SlabGeometry, minstd_uniform, sampled

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def co():
    return COracle()


@pytest.fixture(scope="module")
def gold():
    with open(os.path.join(HERE, "golden", "heffte_ref_vectors.json")) as f:
        return json.load(f)


def _oracle_spectrum(co, A, P, numpy_twin=False):
    n0, n1, n2 = A.shape
    g = SlabGeometry(n0, n1, n2, P)
    ns = NumpySlab(n0, n1, n2, P)
    b1 = ns.scatter_input(A)
    b2 = [np.zeros_like(b) for b in b1]
    if numpy_twin:
        ns.execute(b1, b2, FORWARD)
    else:
        co.slab_execute(g, b1, b2, FORWARD)
    return ns.gather_forward_output(b2)


def test_restated_oracles_reproduce_the_reference_librarys_spectra(co, gold):
    assert "heFFTe 210" in gold["library"]
    for case in gold["cases"]:
        n0, n1, n2 = case["shape"]
        A = np.asarray(case["input_real"], dtype=np.float64).astype(np.complex128).reshape(n0, n1, n2)
        sp = np.asarray(case["spectrum"])
        S = (sp[:, 0] + 1j * sp[:, 1]).reshape(n0, n1, n2)
        for P in sorted({1, case["ranks"]}):
            for twin in (False, True):
                got = _oracle_spectrum(co, A, P, twin)
                assert np.abs(got - S).max() <= 1e-13 * np.log2(A.size) * np.abs(S).max(), (case["shape"], P, twin)
    # the 2x3x4 box of 1..24 (test_units_nompi.cpp:92-98): its DC bin is the sum 300
    s0 = np.asarray(gold["cases"][0]["spectrum"][0])
    assert abs(s0[0] - 300.0) < 1e-12 and abs(s0[1]) < 1e-12


@pytest.fixture(scope="module")
def rec():
    return np.load(os.path.join(HERE, "golden", "ref_samples.npz"))


HEFFTE_LIVE = [(8, 16, 4, 1, "alltoallv"), (16, 16, 16, 2, "p2p_plined"), (10, 9, 4, 3, "p2p"), (9, 10, 4, 3, "alltoall"), (12, 10, 24, 4, "p2p_plined"),
               (24, 16, 16, 8, "alltoallv"), (64, 64, 64, 8, "p2p_plined")]


@pytest.mark.parametrize("n0,n1,n2,P,alg", HEFFTE_LIVE)
def test_live_reference_library_agrees_with_the_oracle(co, rec, n0, n1, n2, P, alg):
    assert int(rec["heffte/version"]) == 210
    key = f"heffte/{HEFFTE_LIVE.index((n0, n1, n2, P, alg))}"
    vals, _ = minstd_uniform(n0 * n1 * n2, 4242) if n0 * n1 * n2 <= 8192 else (np.random.default_rng(3).random(n0 * n1 * n2), 0)
    A = (vals + 1j * np.roll(vals, 7)).reshape(n0, n1, n2)
    assert np.array_equal(A.reshape(-1)[:4], rec[key + "/input_head"]), "the recorded input is not the one regenerated here"
    S, B = rec[key + "/forward,backward"]
    got = _oracle_spectrum(co, A, P)
    assert np.abs(sampled(got, S.size) - S).max() <= 1e-13 * np.log2(A.size) * np.abs(got).max()
    # backward: the oracle's unnormalised inverse (3dmpifft_opt leaves normalize=0) equals heFFTe's scale::none backward
    g = SlabGeometry(n0, n1, n2, P)
    ns = NumpySlab(n0, n1, n2, P)
    b1 = []
    for q in range(P):
        b = np.zeros(g.max_count(q), dtype=np.complex128)
        blk = got[:, q * g.yd: q * g.yd + g.n1l(q), :].transpose(1, 2, 0).reshape(-1)
        b[: blk.size] = blk
        b1.append(b)
    b2 = [np.zeros_like(b) for b in b1]
    co.slab_execute(g, b1, b2, BACKWARD)
    back = ns.gather_natural(b2)
    assert np.abs(sampled(back, B.size) - B).max() <= 1e-13 * np.log2(A.size) * np.abs(back).max()
    assert np.abs(B / A.size - sampled(A, B.size)).max() <= 1e-11      # heFFTe's own round-trip tolerance (test_common.h:136-140)


def test_live_reference_float_precision(rec):
    rng = np.random.default_rng(5)
    A = (rng.random((16, 12, 8)) + 1j * rng.random((16, 12, 8))).astype(np.complex64)
    assert np.array_equal(A.reshape(-1)[:4], rec["heffte/float/input_head"])
    S = rec["heffte/float/forward"]
    want = np.fft.fftn(A.astype(np.complex128))
    assert S.dtype == np.complex64 and np.abs(S - sampled(want, S.size)).max() / np.abs(want).max() <= 5e-6
