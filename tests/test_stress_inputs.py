"""CPU: the adversarial windows of tests/stress_inputs.py are well posed (both fp64 oracles give the same answer), reach
the limits they were built for, and the oracles follow the reference's own work() on them
(tests/golden/reference_source/stress.npz, written by tests/golden/make_reference_golden.py)."""
import os
import re

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import music_oracle as mo

import helpers
import stress_inputs as si

CSRC = os.path.join(helpers.ROOT, "gr-baz_b200", "csrc")


def _constant(header, pattern):
    with open(os.path.join(CSRC, header)) as f:
        return re.search(pattern, f.read()).group(1)


def test_generator_constants_follow_the_kernels():
    """the limits the families are built around are the kernels' own"""
    assert int(_constant("music_eig4p.cuh", r"constexpr int EIGP_MAXSQ = (\d+);")) == si.EIGP_MAXSQ
    for header in ("music_eig4p.cuh", "music_fused8.cuh"):
        assert float(_constant(header, r"const bool pass = f >= ([0-9.]+) \* \(t \* t\);")) == si.RANK_ONE
    assert int(_constant("music_fused.cuh", r"constexpr int FZ_CMAX = (\d+);")) == si.FZ_CMAX
    assert float(_constant("music_fused.cuh", r"constexpr float FZ_B = ([0-9.e+-]+)f;")) == si.FZ_B
    scan_warps = int(_constant("music_fused.cuh", r"constexpr int FZ_SCAN_WARPS = (\d+);"))
    mpw = int(_constant("music_fused.cuh", r"constexpr int FZ_MPW = (\d+);"))
    assert 16 * scan_warps * mpw == si.FZ_BINS


def test_squaring_limit():
    """12 squarings including the extra one after the rank-one test: l2/l1 must be below ~0.9896"""
    lim = si.squaring_limit()
    assert 0.9895 < lim < 0.9897
    r = lim ** (2 ** (si.EIGP_MAXSQ - 1))
    assert abs((1 + r * r) / (1 + r) ** 2 - si.RANK_ONE) < 1e-15


@pytest.mark.parametrize("key", sorted(si.CASES) + sorted(si.ROUTE_CASES))
def test_windows_are_well_posed(key):
    """numpy/LAPACK and C/Jacobi oracles agree on every finite window: bins identical, P to 1e-9 (measured <= 3.3e-10,
    on the noiseless windows a thousandth of a bin off a grid row)"""
    cfg, table, x = si.case(key)
    m, n = cfg["m"], cfg["n"]
    c = co.work_batch(x, m, n, table)
    finite = ~si.nonfinite_windows(x)
    assert finite.sum() >= x.shape[0] // 2
    for w in np.nonzero(finite)[0]:
        p = mo.work(x[w], m, n, table)
        assert np.array_equal(p["bins"], c["bins"][w]), (key, w)
        assert np.all(c["bins"][w] >= 0), (key, w)
        assert helpers.rel_err(c["P"][w], p["P"]) <= 1e-9, (key, w)
    if si.FAMILY.get(key) == "nonfinite":  # the non-finite windows: nothing is ever inserted
        assert np.all(c["bins"][~finite] == -1) and np.all(c["levels"][~finite] == 0) and np.all(c["angles"][~finite] == 0)


@pytest.mark.parametrize("m", [4, 8])
def test_gap_family_straddles_the_squaring_limit(m):
    cfg, _, x = si.case("gap_m%d" % m)
    ratio = si.achieved_gap(cfg, x)
    lim = si.squaring_limit()
    below, above = ratio < lim, ratio > lim
    assert below.sum() >= 2 and above.sum() >= 2, ratio
    assert ratio.min() >= 0.949 and ratio.max() <= 0.9995, ratio
    # clear of the limit, so that which solver handles a window does not hang on rounding: the ratio of the last
    # squaring step, (l2/l1)^2048, is at least 10x away from the rank-one threshold
    p = 2.0 ** (si.EIGP_MAXSQ - 1)
    rstar = lim ** p
    assert np.all(np.abs(np.log10(ratio ** p / rstar)) >= 1.0), ratio ** p / rstar


@pytest.mark.parametrize("key", ["screen_36000", "screen_100000"])
def test_screen_family_overflows_the_candidate_list(key):
    """more than FZ_CMAX bins of a non-flat spectrum certainly pass the screen (admission band from the oracle's
    principal eigenvector and the screen error bound)"""
    cfg, table, x = si.case(key)
    counts = []
    for w in x:
        _, V = np.linalg.eigh(mo.covariance(w, 4))
        counts.append(si.screen_survivors(table, V[:, -1]))
    assert sum(c > si.FZ_CMAX for c in counts) >= 4, counts
    assert sum(c <= si.FZ_CMAX for c in counts) >= 1, counts  # and windows that keep the candidate list
    assert cfg["resolution"] > si.FZ_BINS


@pytest.mark.parametrize("key", sorted(si.CASES))
def test_oracles_follow_the_reference_on_stress_windows(key):
    cfg, table, x = si.case(key)
    ref = helpers.reference_result("stress", key, x)
    c = co.work_batch(x, cfg["m"], cfg["n"], table, want_spectrum=True)
    finite = ~si.nonfinite_windows(x)
    assert np.array_equal(c["angles"], ref["angles"])
    assert helpers.rel_err(c["levels"][finite], ref["levels"][finite]) <= 1.2e-7
    sp = c["spectrum"][:, ref["spec_idx"]]
    assert helpers.rel_err(sp[finite], ref["spectrum"][finite]) <= 1.2e-7
    # a non-finite sample: the reference's eig_sym sees NaN / Inf in R and never inserts a peak; this project specifies
    # the same outcome (angle 0, level 0, bin -1; DESIGN.md section 2)
    assert np.all(ref["angles"][~finite] == 0) and np.all(ref["levels"][~finite] == 0)
    assert np.all(c["levels"][~finite] == 0) and np.all(c["bins"][~finite] == -1)
