"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/dfft.h
declares, slab bookkeeping matches the oracle's restatement of the reference, and the process-per-GPU
bootstrap path works over a world_size-2 gloo group (no compute calls: there is no GPU here)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import distributedfft_b200 as dfft
from oracle import BACKWARD, FORWARD, COracle, SlabGeometry, proper_device_num

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dfft.h")).read()
    names = set(re.findall(r"\b(dfft_[a-z0-9_]+)\s*\(", hdr))
    names -= {"dfft_allgather_fn"}
    assert len(names) >= 25
    L = dfft.lib()
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing


def test_supported_lengths_cover_baseline_configs():
    for prec in (dfft.DOUBLE, dfft.FLOAT):
        ls = dfft.supported_lengths(prec)
        for n in (64, 512, 768, 1024):
            assert n in ls
        assert ls == sorted(ls)


def test_slab_bookkeeping_matches_oracle():
    co = COracle()
    for (n0, n1, n2, P) in [(512, 512, 512, 8), (10, 9, 4, 3), (9, 10, 4, 3), (64, 64, 64, 4), (768, 768, 768, 8), (7, 12, 4, 3)]:
        g = SlabGeometry(n0, n1, n2, P)
        for d in range(P):
            assert dfft.getMaxDataCount(n0, n1, n2, P, d == P - 1) == co.lib.oracle_max_data_count(n0, n1, n2, P, int(d == P - 1))
            alloc, ln0, s0, ln1, s1 = dfft.fft_mpi_local_size_3d(n0, n1, n2, P, d)
            assert (alloc, ln0, s0, ln1, s1) == (g.max_count(d), g.n0l(d), d * g.xd, g.n1l(d), d * g.yd)
            for direction in (FORWARD, BACKWARD):
                mine = dfft.exchange_table(n0, n1, n2, P, d, direction)
                ref = co.exchange_table(n0, n1, n2, P, d, direction)
                for k in ("scount", "soffset", "rcount", "roffset"):
                    assert mine[k] == list(ref[k]), (k, d, direction)


def test_slab_bookkeeping_random_geometries_match_oracle():
    """300 random (N0, N1, N2, P <= 8) incl. every kind of short last slab: counts, local sizes and the four exchange-table
    columns (api.cpp:84-133, 289-316) equal the oracle's restatement for every device and both directions."""
    import numpy as np
    co = COracle()
    rng = np.random.default_rng(2024)
    checked = 0
    for _ in range(300):
        P = int(rng.integers(1, 9))
        n0, n1, n2 = (int(rng.integers(1, 97)) for _ in range(3))
        splittable = all((P - 1) * -(-n // P) < n for n in (n0, n1))
        if not splittable:          # the reference never gets here: fft_mpi_init lowers the device count first (api.cpp:232-272)
            continue
        g = SlabGeometry(n0, n1, n2, P)
        for d in range(P):
            assert dfft.getMaxDataCount(n0, n1, n2, P, d == P - 1) == co.lib.oracle_max_data_count(n0, n1, n2, P, int(d == P - 1))
            assert dfft.fft_mpi_local_size_3d(n0, n1, n2, P, d) == (g.max_count(d), g.n0l(d), d * g.xd, g.n1l(d), d * g.yd)
            for direction in (FORWARD, BACKWARD):
                mine = dfft.exchange_table(n0, n1, n2, P, d, direction)
                ref = co.exchange_table(n0, n1, n2, P, d, direction)
                for k in ("scount", "soffset", "rcount", "roffset"):
                    assert mine[k] == list(ref[k]), (n0, n1, n2, P, k, d, direction)
        checked += 1
    assert checked > 150


def test_fft_mpi_init_device_policy(n_gpus):
    """getProperDeviceNum (api.cpp:232-272): the wanted count is clamped to the GPUs present (api.cpp:236-239); without a
    GPU it is not clamped."""
    def usable(w):
        return min(w, n_gpus) if n_gpus else w
    for n0, w in ((512, 8), (10, 4), (9, 4), (5, 4), (7, 3)):
        tot, loc, counts = dfft.fft_mpi_init([n0, 64, 4], w)
        assert tot == loc == proper_device_num(n0, usable(w))
        g = SlabGeometry(n0, 64, 4, tot)
        assert counts == [g.in_count(p) for p in range(tot)]
    if usable(4) == 4:
        with pytest.raises(dfft.DfftError):
            dfft.fft_mpi_init([8, 3, 4], 4)   # N1=3 over 4 devices leaves an empty y-slab
    else:
        assert dfft.fft_mpi_init([8, 3, 4], 4)[0] == proper_device_num(8, usable(4))


def test_plan_rejects_bad_arguments_without_touching_a_gpu():
    with pytest.raises(dfft.DfftError, match="unsupported transform length"):
        dfft.fft_mpi_plan_dft_c2c_3d(17, 16, 16, 1, 2, None, 0, 1, FORWARD)
    with pytest.raises(dfft.DfftError, match="communicator"):
        dfft.fft_mpi_plan_dft_c2c_3d(16, 16, 16, 1, 2, None, 0, 2, FORWARD)
    with pytest.raises(dfft.DfftError, match="empty last slab"):
        c = dfft.LocalComm(4)
        try:
            dfft.fft_mpi_plan_dft_c2c_3d(6, 16, 16, 1, 2, c, 0, 4, FORWARD)
        finally:
            c.destroy()


def test_local_comm_allgather_threads():
    import threading
    P = 4
    comm = dfft.LocalComm(P)
    out = [None] * P

    def w(r):
        out[r] = dfft.comm_allgather(comm, r, bytes([r]) * 64)

    th = [threading.Thread(target=w, args=(r,)) for r in range(P)]
    [t.start() for t in th]; [t.join() for t in th]
    for r in range(P):
        assert out[r] == [bytes([q]) * 64 for q in range(P)]
    comm.destroy()


WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
import distributedfft_b200 as dfft
from oracle import SlabGeometry
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
def ag(b):
    out = [None] * world
    dist.all_gather_object(out, b)
    return out
comm = dfft.BootstrapComm(rank, world, ag)
# 1. the bootstrap all-gather used for IPC handles / NCCL id (64- and 128-byte payloads)
for size in (64, 128):
    got = dfft.comm_allgather(comm, rank, bytes([rank + 1]) * size)
    assert got == [bytes([q + 1]) * size for q in range(world)], got
# 2. every rank's exchange table agrees with its peers' (scount[r] on me == rcount[me] on r)
n0, n1, n2 = 10, 9, 4
for direction in (1, -1):
    mine = dfft.exchange_table(n0, n1, n2, world, rank, direction)
    tabs = [None] * world
    dist.all_gather_object(tabs, mine)
    for r in range(world):
        assert mine["scount"][r] == tabs[r]["rcount"][rank]
        assert mine["rcount"][r] == tabs[r]["scount"][rank]
    g = SlabGeometry(n0, n1, n2, world)
    assert sum(mine["scount"]) == (g.in_count(rank) if direction == 1 else g.out_count(rank))
comm.destroy()
dist.barrier()
dist.destroy_process_group()
sys.stdout.write("rank %d ok\n" % rank); sys.stdout.flush()
'''


def test_bootstrap_comm_world2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29571", str(script), ROOT], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout


def test_length_policy_matches_the_reference_generator():
    """Lengths: tuned table, run-time-scheduled 2..13-smooth lengths with the radix policy restated in oracle_fft.c from
    templateFFT.cpp:3956-3963 (factor over 2..13), :4540-4550 (merge 2s into 8s then 4s), :4580-4588 (descending order),
    everything else rejected.  (Against the EXECUTED generator -- tests/test_oracle_ref3d.py -- that restatement is exact for
    powers of 2, 3, 5, 7; for mixed lengths the generator merges the 2s only when its register counts allow it.)"""
    co = COracle()
    for n in (512, 768, 1024, 64, 100):
        assert dfft.length_kind(n) == 2 and dfft.length_kind(n, dfft.FLOAT) == 2
        assert int(np.prod(dfft.length_schedule(n))) == n
    for n in (2, 3, 5, 7, 11, 13, 15, 30, 77, 143, 360, 1001, 2187, 3000, 3125, 6400, 6144):
        assert dfft.length_kind(n) == 1, n
        assert dfft.length_schedule(n) == co.radix_schedule(n), n
    for n in (17, 19, 34, 6561, 8192, 1 << 21):
        assert dfft.length_kind(n) == 0 and dfft.length_schedule(n) == []
    assert dfft.length_kind(8192, dfft.FLOAT) == 1 and dfft.length_kind(12800, dfft.FLOAT) == 1 and dfft.length_kind(16384, dfft.FLOAT) == 0


@pytest.mark.parametrize("planes,rows,GA,GBk,GXk,K,lag", [(64, 64, 128, 16, 16, 4, 3), (5, 7, 3, 2, 1, 2, 2), (8, 3, 4, 1, 5, 8, 100), (1, 1, 1, 1, 1, 1, 1),
                                                      (6, 6, 2, 3, 3, 1, 2)])
def test_single_kernel_forward_ticket_order(planes, rows, GA, GBk, GXk, K, lag):
    """The ticket order of the single-kernel forward path (fft_fused3_kernel) must hand out every Z, Y and X tile
    exactly once, and every dependency must have a lower ticket: Z tiles of a plane before its Y tiles, all Y tiles of
    part k (on this device) before any X tile of part k."""
    import ctypes
    L = dfft.lib()
    out = (ctypes.c_longlong * 4)()
    total = L.dfft_debug_fused3_order(planes, rows, GA, GBk, GXk, K, lag, -1, out)
    assert total == planes * (GA + GBk * K) + rows * GXk * K
    seen = set()
    last_z = {}        # plane -> highest ticket of its Z tiles
    last_y = {}        # part -> highest ticket of its Y tiles
    first_y = {}       # plane -> lowest ticket of its Y tiles
    first_x = {}       # part -> lowest ticket of its X tiles
    for t in range(total):
        assert L.dfft_debug_fused3_order(planes, rows, GA, GBk, GXk, K, lag, t, out) == total
        role, part, plane, idx = (int(x) for x in out)
        key = (role, part, plane, idx)
        assert key not in seen, key
        seen.add(key)
        if role == 0:
            assert 0 <= plane < planes and 0 <= idx < GA and part == 0
            last_z[plane] = t
        elif role == 1:
            assert 0 <= plane < planes and 0 <= idx < GBk and 0 <= part < K
            last_y[part] = t
            first_y.setdefault(plane, t)
        else:
            assert role == 2 and 0 <= idx < rows * GXk and 0 <= part < K
            first_x.setdefault(part, t)
    assert len(seen) == total
    for plane in range(planes):
        assert last_z[plane] < first_y[plane]
    for part in range(K):
        assert last_y[part] < first_x[part]
