"""CPU check that tests/kernel_matrix.py runs every kernel the library can launch.

Every case of the matrix is planned with DRY_RUN (no CUDA call; dfft_execute records the passes it would launch, see
tests/test_dry_run.py) and executed in each of its directions.  The recorded passes name the SizeEntry they come from (length,
precision) and the instantiation (pass kind, fused t0 kind with its chunk flags, kernel-chain link), and their union must
cover every (precision, length, kind) of the library: the 8 pass kinds of every tuned length in dfft.supported_lengths and
the fused t0 kinds it has (kernel_matrix.FUSED_ABSENT lists the ones too large for one CTA's shared memory), every
radix of the generic kernel in each of its single-device launchers, the chunked generic launchers, and the chain link
wherever a two-device cube plan of that length runs one.  The TMA kernels are not recorded by dry runs; their table is
checked against dfft_kernels_tma.cu, and the GPU tests assert Plan.tma_mask for each case."""
import os
import re

import pytest

import distributedfft_b200 as dfft
import kernel_matrix as km

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PASS_KINDS = ["Z", "Y", "Y_CO", "Y_CI", "XF", "XB", "XB_CO", "XF_TW"]
TWO_DEVICE_KINDS = {"Y_CO", "Y_CI", "XB_CO", "fusedZY_CO", "fusedYZ_CI", "fused_yx"}
GENERIC_RADICES = [2, 3, 4, 5, 7, 8, 11, 13]


def kinds_of(ops, chain):
    """(kind, N) of every kernel launch in one plan's recorded passes"""
    out = []
    i = 0
    while i < len(ops):
        o = ops[i]
        name = o["op"]
        if name == "fusedY":   # the fused t0 kernel records its two roles (fusedZ, fusedY); the Y role names the kind
            kind = ("fusedZY" if o["phase"] == 0 else "fusedYZ") + ("_CO" if "co" in o else "_CI" if "ci" in o else "")
            out.append((kind, o["N"]))
        elif chain and name == "Y_CO" and i + 1 < len(ops) and ops[i + 1]["op"] == "XF":
            out.append(("fused_yx", o["N"]))   # one two-role kernel: Y pass of part k + X pass of part k-1
            i += 2
            continue
        elif name == "ovlY":   # the single-kernel forward (fft_fused3_kernel)
            out.append(("fused3", o["N"]))
        elif name in PASS_KINDS:
            out.append((name, o["N"]))
        i += 1
    return out


def dry_case(case, monkeypatch):
    """[(precision, kind, N)] recorded by every device's plan of `case`, and the plan properties per device and direction"""
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    n0, n1, n2 = case.shape
    got, props = [], []
    for direction in case.directions:
        plans = [dfft.fft_mpi_plan_dft_c2c_3d(n0, n1, n2, 1 << 40, 2 << 40, None, d, case.P, direction, case.precision,
                                              case.flags | dfft.DRY_RUN) for d in range(case.P)]
        for p in plans:
            p.execute()
            got += [(case.precision, k, n) for k, n in kinds_of(p.recorded_ops(), p.pipeline_chain)]
            props.append((direction, {"fused": p.fused, "pipeline_chain": p.pipeline_chain, "exchange": p.exchange}))
            p.destroy()
    for k, _ in case.env:
        monkeypatch.delenv(k)
    return got, props


def four_step_kinds(precision, n):
    ops = dfft.lines_ops(n, 1, km.four_step_lines(n), km.four_step_lines(n), n, n, dfft.FORWARD, precision)
    return [(precision, o["op"], o["N"]) for o in ops]


def cube_lengths(precision, flags, has):
    """tuned lengths whose forward two-device P2P cube plan with `flags` satisfies has(plan)"""
    out = []
    for L in km.TUNED:
        p = dfft.fft_mpi_plan_dft_c2c_3d(L, L, L, 1 << 40, 2 << 40, None, 0, 2, dfft.FORWARD, precision, dfft.EXCHANGE_P2P | flags | dfft.DRY_RUN)
        p.execute()
        if has(p):
            out.append(L)
        p.destroy()
    return out


def chain_lengths(precision):
    return cube_lengths(precision, dfft.FORCE_PIPELINE, lambda p: p.pipeline_chain)


def fused3_lengths(precision):
    return cube_lengths(precision, dfft.OVERLAP_X, lambda p: p.overlapped)


def required(precision):
    req = set()
    for L in dfft.supported_lengths(precision):
        req |= {(precision, k, L) for k in PASS_KINDS}
        req |= {(precision, k, L) for b, k in enumerate(km.FUSED_NAMES[:4]) if dfft.fused_kinds(L, precision) >> b & 1}
    req |= {(precision, "fused_yx", L) for L in chain_lengths(precision)}
    req |= {(precision, "fused3", L) for L in fused3_lengths(precision)}
    req |= {(precision, k, f"generic/{r}") for k in ("Z", "Y", "XF", "XB") for r in GENERIC_RADICES}
    req |= {(precision, k, "generic") for k in ("Y_CO", "Y_CI", "XB_CO", "XF_TW")}
    return req


def excluded(precision):
    """explicit exclusions: (precision, kind, N) -> reason"""
    ex = {(precision, "fused3", L): km.EXCLUDED["fused3"] for L in fused3_lengths(precision)}
    ex.update({(precision, "fused_yx", L): km.EXCLUDED["fused_yx"] for L in chain_lengths(precision) if L ** 3 > km.CHAIN_MAX_ELEMENTS})
    return ex


@pytest.mark.parametrize("precision", [km.D, km.F], ids=["f64", "f32"])
def test_fused_kernels_left_out_are_the_listed_ones(precision):
    """kernel_matrix.FUSED_ABSENT names every multi-role kernel a tuned entry lacks (roles too large for one CTA's shared
    memory); a plan of such a length that wants fusion runs the passes as separate kernels (the zy-fused / p2p cases expect so)"""
    for L in km.TUNED:
        m = dfft.fused_kinds(L, precision)
        absent = tuple(b for b in range(6) if not m >> b & 1)
        assert absent == km.FUSED_ABSENT[precision].get(L, ()), (L, [km.FUSED_NAMES[b] for b in absent])


def normalise(rec):
    """tuned records stay (precision, kind, N); generic ones become (precision, kind, 'generic/<radix>') per radix and
    (precision, kind, 'generic')"""
    out = set()
    for prec, kind, n in rec:
        if dfft.length_kind(n, prec) == 2:
            out.add((prec, kind, n))
        else:
            out.add((prec, kind, "generic"))
            out |= {(prec, kind, f"generic/{r}") for r in dfft.length_schedule(n, prec)}
    return out


@pytest.fixture(scope="module")
def coverage():
    mp = pytest.MonkeyPatch()
    cov = {1: set(), 2: set()}   # by device count of the covering case
    props = []
    try:
        for case in km.single_device_cases() + km.two_device_cases():
            rec, pr = dry_case(case, mp)
            cov[case.P] |= normalise(rec)
            props.append((case, pr))
    finally:
        mp.undo()
    for prec in (km.D, km.F):
        for table in (km.FOUR_STEP[prec], km.FOUR_STEP_GENERIC[prec]):
            for n in table.values():
                cov[1] |= normalise(four_step_kinds(prec, n))
    return cov, props


def test_the_tuned_length_table_is_the_librarys():
    for prec in (km.D, km.F):
        assert sorted(dfft.supported_lengths(prec)) == sorted(km.TUNED), "kernel_matrix.TUNED is out of date"
        for L in km.GENERIC:
            assert dfft.length_kind(L, prec) == 1, (prec, L)


@pytest.mark.parametrize("precision", [km.D, km.F], ids=["f64", "f32"])
def test_every_instantiation_has_a_case(coverage, precision):
    cov, _ = coverage
    have = cov[1] | cov[2]
    req = required(precision)
    ex = excluded(precision)
    missing = sorted(req - have - set(ex), key=str)
    assert not missing, "no case in tests/kernel_matrix.py runs: " + ", ".join(f"({km.PREC_NAME[p]}, {n}, {k})" for p, k, n in missing)
    # an exclusion that a case covers after all is stale
    assert not (set(ex) & have), sorted(set(ex) & have, key=str)


@pytest.mark.parametrize("precision", [km.D, km.F], ids=["f64", "f32"])
def test_kinds_that_only_two_device_cases_run(coverage, precision):
    """the chunked kinds, the chunked fused t0 kernels and the chain link run only with P >= 2; everything else on one device"""
    cov, _ = coverage
    only2 = {(k, n) for p, k, n in cov[2] - cov[1] if p == precision}
    assert {k for k, _ in only2} == TWO_DEVICE_KINDS
    assert not {k for p, k, n in cov[1] if p == precision} & TWO_DEVICE_KINDS


def test_cases_take_the_path_they_name(coverage):
    """the plan properties a case expects (fused, chain, exchange) hold for its dry plans too; tma_mask is GPU-only"""
    _, props = coverage
    for case, pr in props:
        for direction, d in pr:
            for k, _ in case.expect:
                if k != "tma_mask":
                    v = km.expected(case, k, direction)
                    assert d[k] == v, (case.id, direction, k, d[k], v)


@pytest.mark.parametrize("precision", [km.D, km.F], ids=["f64", "f32"])
def test_four_step_first_factors(precision):
    """make_four_step picks the pinned first factor for every pinned length, and no single kernel covers that length"""
    for first, n in list(km.FOUR_STEP[precision].items()) + list(km.FOUR_STEP_GENERIC[precision].items()):
        assert dfft.length_kind(n, precision) == 0, n
        ops = four_step_kinds(precision, n)
        assert [k for _, k, _ in ops] == ["XF_TW", "Y"] and ops[0][2] == first, (n, ops)


def test_tma_table_matches_the_source():
    """kernel_matrix.TMA lists exactly the make_tma_entry lines of dfft_kernels_tma.cu (length, precision, C, default modes)"""
    with open(os.path.join(ROOT, "distributedfft_b200", "csrc", "dfft_kernels_tma.cu")) as f:
        src = f.read()
    pat = re.compile(r"make_tma_entry<Sched<(\d+)[^>]*>,\s*(double|float),\s*(\d+)>\(([ZYX |]+)\)")
    found = sorted((int(n), km.D if t == "double" else km.F, int(c), "".join(sorted(m.replace("|", "").split())))
                   for n, t, c, m in pat.findall(src))
    assert len(found) == len(km.TMA) == 7
    assert found == sorted((n, p, c, "".join(sorted(m))) for n, p, c, m in km.TMA)


def test_every_tma_mode_of_every_entry_has_a_forced_case():
    need = {(n, p, bit) for n, p, _, _ in km.TMA for bit in range(3)}
    have = set()
    for case in km.single_device_cases():
        if ("DFFT_TMA", "2") not in case.env:
            continue
        mask = dict(case.expect)["tma_mask"]
        n0, n1, n2 = case.shape
        for bit, n in ((0, n2), (1, n1), (2, n0)):
            if mask >> bit & 1:
                have.add((n, case.precision, bit))
    assert need <= have, sorted(need - have)


def test_the_comparison_rejects_what_it_should():
    """kernel_matrix.check at the fp64 / fp32 bounds: an exact spectrum from another FFT passes, so does an fp32 FFT against the
    fp32 bound; two swapped adjacent bins, an fp64 spectrum rounded to fp32 (against the fp64 bound) and x-lines offset by one
    row fail."""
    import numpy as np
    import scipy.fft
    shape = (12, 10, 24)
    N = int(np.prod(shape))
    rng = np.random.default_rng(5)
    A = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    ref = np.fft.fftn(A).transpose(1, 2, 0)                 # [y][z][x], as the plan lays it out
    km.check(scipy.fft.fftn(A).transpose(1, 2, 0), ref, km.D, N, "scipy fp64")
    A32 = A.astype(np.complex64)
    km.check(scipy.fft.fftn(A32).transpose(1, 2, 0), np.fft.fftn(A32.astype(np.complex128)).transpose(1, 2, 0), km.F, N, "scipy fp32")
    swapped = ref.copy()
    swapped[3, 4, [7, 8]] = swapped[3, 4, [8, 7]]
    rounded = ref.astype(np.complex64).astype(np.complex128)
    shifted = np.roll(ref.reshape(-1, shape[0]), 1, axis=0)  # every x-line moved to the next row
    for bad, prec, what in ((swapped, km.D, "swapped bins"), (swapped, km.F, "swapped bins"), (rounded, km.D, "rounded to fp32"),
                            (shifted, km.D, "x-lines offset by one row"), (shifted, km.F, "x-lines offset by one row")):
        with pytest.raises(AssertionError):
            km.check(bad, ref, prec, N, what)
        assert km.rel_err(bad, ref) > 3 * km.bound(prec, N), what
