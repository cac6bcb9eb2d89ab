"""bench.py: the reference arm (the one arm that runs without a GPU) prints one JSON line with the contract's keys; the
arguments are checked; on a GPU, --dump-outputs writes the spectrum the timed steps computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "64", "--steps", "3", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "GFlops/s" and d["higher_is_better"] is True and d["value"] > 0
    # "reference" = the reference tree's heFFTe from oracle/_ref (built from the reference sources where they are); "port" only
    # when that library is absent
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libheffte_ref.so"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "64x64x64" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--size", "64", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and not any(l.startswith("{") for l in r.stdout.splitlines())


def test_arguments_are_checked():
    for extra, msg in ((["--steps", "0"], "--steps must be at least 1"), (["--impl", "reference", "--dump-outputs", "x"], "--dump-outputs")):
        r = subprocess.run([sys.executable, BENCH] + extra, capture_output=True, text=True, timeout=60)
        assert r.returncode == 2 and msg in r.stderr, r.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_spectrum_of_the_timed_steps(tmp_path):
    """Two runs with different step counts dump the same spectrum, and it is the forward transform of bench.py's input
    (U(0,1) real and imaginary parts from torch's CUDA generator seeded 4242), in the [y][z][x] layout of one device."""
    import torch
    n = 64
    dumps = []
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, BENCH, "--size", str(n), "--steps", str(steps), "--warmup", "1", "--no-cpu", "--no-e2e", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == steps
        assert sorted(os.listdir(d)) == ["spectrum_rank0.npy"]
        dumps.append(np.load(d / "spectrum_rank0.npy"))
    assert dumps[0].dtype == np.float64 and dumps[0].shape == (n ** 3, 2)
    assert np.array_equal(dumps[0], dumps[1])
    gen = torch.Generator(device="cuda"); gen.manual_seed(4242)
    a = torch.empty(n ** 3, dtype=torch.complex128, device="cuda")
    torch.view_as_real(a).uniform_(0.0, 1.0, generator=gen)
    want = np.fft.fftn(a.cpu().numpy().reshape(n, n, n)).transpose(1, 2, 0).reshape(-1)
    got = dumps[0][:, 0] + 1j * dumps[0][:, 1]
    assert np.abs(got - want).max() <= 1e-12 * 18 * np.abs(want).max()
