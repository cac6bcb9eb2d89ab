"""The instantiation matrix: 3-D plan cases (and long-line lengths) that together run every kernel the library ships.

Each tuned length has one SizeEntry per precision (dfft_kernels_f64.cu, dfft_kernels_f32.cu) holding separate template
instantiations -- 8 pass kinds (Z, Y, Y_CO, Y_CI, XF, XB, XB_CO, XF_TW), 4 fused t0 kernels (ZY, ZY_CO, YZ, YZ_CI) and the
kernel-chain link fused_yx -- each with its own tile width, thread map and ragged-tile path.  Lengths without a tuned entry
run on the run-time-scheduled generic kernel (dfft_kernels_generic.cu), and seven lengths have TMA-ring kernels
(dfft_kernels_tma.cu) in four modes.  The cases below are chosen so that every one of them runs at least once:

  * X passes: (L, 3, 135).  135 = 27 * 5 is odd and wider than every tuned X tile, so X tiles are ragged, several per row.
  * Z / Y and fused t0: (5, L, L), (2, L, L) for 2048 and 4096; default flags (two sweeps), FORCE_FUSE, NO_TMA.
  * every TMA mode of every TMA entry under DFFT_TMA=2 (modes the entry's `use` mask leaves off included), plus shapes that
    mix two TMA entries of one precision.
  * four-step long lines whose first factor (the PK_XF_TW pass) is every tuned length.
  * generic lengths covering every generic radix in all three axis positions.
  * two devices: (4, L, L) / (2, L, L) in the default P2P mode (fused), P2P without fusion or pipeline, NCCL, and the kernel
    chain on P = 2 cubes.

tests/test_kernel_matrix_complete.py checks on the CPU (DRY_RUN plans) that the union of these cases covers every
(precision, length, kind) the library can launch; tests/test_gpu_parity.py and tests/test_gpu_multi.py run them against an
fp64 numpy reference with `check` below.
"""
from dataclasses import dataclass

import numpy as np

import distributedfft_b200 as dfft

D, F = dfft.DOUBLE, dfft.FLOAT
PREC_NAME = {D: "f64", F: "f32"}

# the tuned lengths of dfft_kernels_f64.cu / dfft_kernels_f32.cu (both tables hold the same lengths)
TUNED = [4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 768, 384, 192, 96, 48, 24, 12, 6, 9, 10, 100, 125, 49, 243, 1000]

# the TMA table of dfft_kernels_tma.cu: (N, precision, C, modes used by default); Z = TMA_Z, Y = TMA_Y, X = TMA_XF | TMA_XB
TMA = [(512, D, 8, "Y"), (1024, D, 4, "YX"), (256, D, 16, "ZYX"), (768, D, 4, "Y"),
       (512, F, 16, "ZYX"), (1024, F, 8, "YX"), (768, F, 8, "YX")]

# generic (run-time-scheduled) lengths: every generic radix (13, 11, 8, 7, 5, 4, 3, 2) in both precisions
GENERIC = [11, 13, 22, 26, 35, 143, 3000, 3125, 6400]   # 6400: the longest fp64 generic line (two copies of 6400 * 16 bytes = 200 KB)

# Four-step long lines (LinesPlan): length -> first factor, which runs as PK_XF_TW.  make_four_step (dfft_api.cu) tries every
# divisor d with d*d <= 4n, d < n and both d and n/d supported, scores 1000 per tuned factor + 500 / (larger / smaller), and
# keeps the first best d.  Each length is the smallest multiple of its first factor for which the rule picks that factor (and
# that no single kernel covers); test_kernel_matrix_complete.py checks the split through dfft_debug_lines_ops.
FOUR_STEP = {
    D: {4: 7436, 8: 6776, 16: 7280, 32: 7776, 64: 6656, 128: 16384, 256: 65536, 512: 262144, 1024: 1048576, 2048: 4194304, 4096: 16777216,
        768: 589824, 384: 147456, 192: 36864, 96: 9216, 48: 6480, 24: 6552, 12: 7020, 6: 7098, 9: 6435, 10: 6760, 100: 10000, 125: 15625,
        49: 6468, 243: 59049, 1000: 1000000},
    F: {4: 37268, 8: 14872, 16: 13520, 32: 14560, 64: 15552, 128: 16384, 256: 65536, 512: 262144, 1024: 1048576, 2048: 4194304, 4096: 16777216,
        768: 589824, 384: 147456, 192: 36864, 96: 12960, 48: 13104, 24: 14040, 12: 13068, 6: 13182, 9: 12870, 10: 13310, 100: 13200, 125: 15625,
        49: 12936, 243: 59049, 1000: 1000000},
}
# long lines whose first factor is a generic length (the generic kernel's twiddle epilogue): 6561 = 27 * 243, 19683 = 81 * 243
FOUR_STEP_GENERIC = {D: {27: 6561}, F: {81: 19683}}

# the kernel chain needs a P = 2 cube L^3; above 2^25 elements the whole-spectrum numpy reference is too slow to run per case
# and 2048^3 / 4096^3 do not fit two devices at all.  512^3 fp64 on two devices runs in test_gpu_baseline_configs (C3c-chain).
CHAIN_MAX_ELEMENTS = 1 << 25
# multi-role kernels a tuned entry does not have because their roles together need more than the 227 KB of shared memory one
# CTA may use (make_entry leaves them out; a plan of that length runs the passes as separate kernels).  Bits as
# dfft.fused_kinds: 0 ZY, 1 ZY_CO, 2 YZ, 3 YZ_CI (fused t0), 4 fused_yx (chain link), 5 fused3.
FUSED_ABSENT = {
    D: {2048: (1, 3, 4, 5), 4096: (0, 1, 2, 3, 4, 5)},
    F: {4096: (5,)},
}
FUSED_NAMES = ["fusedZY", "fusedZY_CO", "fusedYZ", "fusedYZ_CI", "fused_yx", "fused3"]


def fused_expect(L, precision, P):
    """(forward, backward) value of plan.fused for a square-plane plan of length L that wants fusion"""
    absent = FUSED_ABSENT[precision].get(L, ())
    return (1 if P > 1 else 0) not in absent, (3 if P > 1 else 2) not in absent


def expected(case, key, direction):
    """the value the case expects of plan property `key` for `direction` (None: not asserted)"""
    v = dict(case.expect).get(key)
    return v[0 if direction == dfft.FORWARD else 1] if isinstance(v, tuple) else v


# kinds the matrix leaves out on purpose, with the reason (test_kernel_matrix_complete.py applies them)
EXCLUDED = {
    "fused3": "DFFT_OVERLAP_X (fft_fused3_kernel) is experimental and off by default (DESIGN.md 5.1)",
    "fused_yx": f"kernel chain of a length whose P = 2 cube exceeds {CHAIN_MAX_ELEMENTS} elements",
}


@dataclass(frozen=True)
class Case:
    shape: tuple
    precision: int
    P: int = 1
    flags: int = 0
    env: tuple = ()              # ((name, value), ...) set while the plans are created and run
    directions: tuple = (dfft.FORWARD, dfft.BACKWARD)
    expect: tuple = ()           # ((property, value), ...): plan.fused, plan.pipeline_chain, plan.tma_mask, plan.exchange;
                                 # a (forward, backward) pair where the two directions differ
    tag: str = ""

    @property
    def id(self):
        s = "x".join(map(str, self.shape))
        return f"{PREC_NAME[self.precision]}-P{self.P}-{s}-{self.tag}"


def tma_entry(n, precision):
    for e in TMA:
        if e[0] == n and e[1] == precision:
            return e
    return None


def default_tma_mask(shape, precision, forced=False):
    """Plan.tma_mask of a one-device plan: bit 0 Z pass (n2), bit 1 Y pass (n1), bit 2 X pass (n0) on the TMA kernel"""
    n0, n1, n2 = shape
    m = 0
    for bit, n, mode, ok in ((0, n2, "Z", lambda C: (n0 * n1) % C == 0), (1, n1, "Y", lambda C: n2 % C == 0), (2, n0, "X", lambda C: n2 % C == 0)):
        e = tma_entry(n, precision)
        if e and (forced or mode in e[3]) and ok(e[2]):
            m |= 1 << bit
    return m


def zy_shape(L):
    return (2, L, L) if L >= 2048 else (5, L, L)


def single_device_cases():
    cases = []
    for prec in (D, F):
        for L in TUNED:
            has_tma = tma_entry(L, prec) is not None
            # X passes (XF forward, XB backward), ragged X tiles
            xs = (L, 3, 135)
            cases.append(Case(xs, prec, expect=(("fused", False), ("tma_mask", 0)), tag="x"))
            if has_tma:
                cases.append(Case(xs, prec, flags=dfft.NO_TMA, expect=(("fused", False), ("tma_mask", 0)), tag="x-notma"))
            # Z / Y passes (two sweeps, TMA where the entry uses it) and the fused t0 kernels
            s = zy_shape(L)
            cases.append(Case(s, prec, expect=(("fused", False), ("tma_mask", default_tma_mask(s, prec))), tag="zy"))
            cases.append(Case(s, prec, flags=dfft.FORCE_FUSE, expect=(("fused", fused_expect(L, prec, 1)),), tag="zy-fused"))
            if has_tma:
                cases.append(Case(s, prec, flags=dfft.NO_TMA, expect=(("fused", False), ("tma_mask", 0)), tag="zy-notma"))
    # every mode of every TMA entry, forced on (DFFT_TMA=2): Z needs (n0 * n1) % C == 0, Y and X need n2 % C == 0
    for N, prec, C, _ in TMA:
        for s in ((4, N, N), (N, 4, 16)):
            cases.append(Case(s, prec, env=(("DFFT_TMA", "2"),), expect=(("fused", False), ("tma_mask", default_tma_mask(s, prec, forced=True))),
                              tag="tma-forced"))
    # two different TMA entries of one precision in one plan (Z on one, X on the other)
    for s, prec in (((256, 16, 512), D), ((768, 8, 512), F), ((1024, 4, 256), D)):
        for env, tag in (((("DFFT_TMA", "2"),), "tma-mixed-forced"), ((), "tma-mixed")):
            cases.append(Case(s, prec, env=env, expect=(("fused", False), ("tma_mask", default_tma_mask(s, prec, forced=bool(env)))), tag=tag))
    # generic kernel: every generic length in all three axis positions
    for prec in (D, F):
        for trio in ((11, 13, 22), (26, 35, 143)):
            for r in range(3):
                cases.append(Case(trio[r:] + trio[:r], prec, expect=(("fused", False), ("tma_mask", 0)), tag="generic"))
        for L in GENERIC[6:]:
            for s in ((L, 4, 6), (6, L, 4), (4, 6, L)):
                cases.append(Case(s, prec, expect=(("fused", False), ("tma_mask", 0)), tag="generic"))
    return cases


def two_device_cases():
    P2P, NCCL = dfft.EXCHANGE_P2P, dfft.EXCHANGE_NCCL
    cases = []
    for prec in (D, F):
        for L in TUNED:
            s = (2, L, L) if L >= 2048 else (4, L, L)
            cases.append(Case(s, prec, 2, P2P, expect=(("fused", fused_expect(L, prec, 2)), ("pipeline_chain", False), ("exchange", P2P)), tag="p2p"))
            cases.append(Case(s, prec, 2, P2P | dfft.NO_FUSE | dfft.NO_PIPELINE, expect=(("fused", False), ("pipeline_chain", False), ("exchange", P2P)),
                              tag="p2p-nofuse"))
            cases.append(Case(s, prec, 2, NCCL, expect=(("fused", False), ("exchange", NCCL)), tag="nccl"))
            cases.append(Case(s, prec, 2, P2P | dfft.FORCE_PIPELINE, expect=(("fused", fused_expect(L, prec, 2)), ("exchange", P2P)), tag="p2p-pipe"))
            # the X axis split over the devices: XB_CO (backward, chunked peer store) and XF of this length
            cases.append(Case((L, 3, 135), prec, 2, P2P, expect=(("fused", False), ("exchange", P2P)), tag="x-p2p"))
            if L ** 3 <= CHAIN_MAX_ELEMENTS:
                # the kernel chain (fft_fused_yx_kernel) needs a cube; cases where the length has no chain are dropped by the
                # completeness test's cross-check, not here, so that a new chain shows up as uncovered
                cases.append(Case((L, L, L), prec, 2, P2P | dfft.FORCE_PIPELINE, directions=(dfft.FORWARD,), expect=(("exchange", P2P),), tag="chain"))
        # generic lengths through the chunked kinds (Y_CO, Y_CI, XB_CO)
        for trio in ((26, 35, 143), (143, 26, 35), (35, 143, 26)):
            cases.append(Case(trio, prec, 2, P2P, expect=(("fused", False), ("exchange", P2P)), tag="generic-p2p"))
    return cases


def four_step_lines(n):
    """lines per four-step case: a few short lines, one long one (the largest, 2^24 points, is 256 MB in fp64)"""
    return max(1, min(3, (1 << 22) // n))


def rel_err(got, ref):
    """max |got - ref| / rms(ref)"""
    got = np.asarray(got).reshape(-1)
    ref = np.asarray(ref).reshape(-1)
    return float(np.abs(got - ref).max() / np.sqrt(np.mean(np.abs(ref) ** 2)))


def bound(precision, n):
    """error bound of a transform of n points (the product of the axis lengths of a 3-D transform)"""
    return (1e-13 if precision == D else 1e-6) * np.log2(max(n, 2))


# worst error / bound seen per precision in this process (printed by the GPU suites)
OBSERVED = {}


def check(got, ref, precision, n, what):
    err = rel_err(got, ref)
    b = bound(precision, n)
    assert err <= b, f"{what}: max|err|/rms(ref) = {err:.3e} > bound {b:.3e}"
    worst = OBSERVED.get(precision)
    if worst is None or err / b > worst[0] / worst[1]:
        OBSERVED[precision] = (err, b, what)
    return err


def report():
    return "; ".join(f"{PREC_NAME[p]}: worst {e:.3e} vs bound {b:.3e} (x{b / e if e else float('inf'):.1f} margin) at {w}"
                     for p, (e, b, w) in sorted(OBSERVED.items()))
