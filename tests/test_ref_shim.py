"""CPU: the oracle restatements against the reference's OWN work() - the reference's lib/baz_music_doa.cc compiled
unmodified against stand-in headers (oracle/ref_shim/armadillo: eig_sym -> LAPACK zheevd, operator* -> zgemm from
scipy's OpenBLAS; lib/gr_shim: GNU Radio / Boost).  Checks that the restatements follow the reference's control flow
exactly: reshape order, noise-subspace selection, the per-step loop, the top-n insertion with its tie rule, the float
casts.  The arithmetic inside Armadillo proper is NOT exercised (that library is absent), so this narrows, but does not
close, the "parity unpinned" gap (DESIGN.md section 2).  What that library returned on these inputs is stored in
tests/golden/reference_source/cpu.npz (tests/golden/make_reference_golden.py), so the checks run without it."""
import numpy as np
import pytest

from gr_baz_b200 import synth
from oracle import c_oracle as co
from oracle import music_oracle as mo

import helpers

FIXTURE = "cpu"

SEEDED = [
    (1, {}, 12), (1, {"n": 2}, 8), (1, {"n": 3}, 8), (1, {"geometry": "ula_y"}, 6),
    (2, {"snapshots": 512}, 6), (4, {"snapshots": 256, "n": 3}, 5), (5, {"snapshots": 256, "resolution": 720}, 4),
    (1, {"m": 6, "geometry": "uca", "n": 2}, 5),
]


def angles_to_bins(ang, K):
    return np.rint(np.asarray(ang, np.float64) * K / 360.0).astype(np.int64)


def golden_key(path):
    return "golden_" + path.split("/")[-1][:-4]


def golden_input(path):
    cfg, _, table, wins, _ = helpers.load_golden(path)
    return cfg, table, wins, np.stack([w["in"] for w in wins])


def seeded_input(base, over, W):
    cfg = synth.config(base, **over)
    return cfg, helpers.table_for(cfg), synth.gen_windows_numpy(cfg, 2024 + base, 0, W)


def mirror_input():
    cfg = synth.config(1, n=2)
    return cfg, helpers.table_for(cfg), synth.gen_windows_numpy(cfg, 77, 0, 10)


def random_small_shapes():
    """(trial, m, n, snaps, K, table, x): small shapes (m 2..9, every valid n, odd grids, single-snapshot windows,
    strong / weak / no signal), one fixed seeded sequence"""
    rng = np.random.default_rng(20260922)
    for trial in range(60):
        m = int(rng.integers(2, 10))
        n = int(rng.integers(1, m))
        snaps = int(rng.choice([1, 2, 3, 7, 16, 33, 64]))
        K = int(rng.choice([7, 12, 45, 90, 360, 721]))
        W = 3
        pos = rng.uniform(-1.5, 1.5, (m, 2))
        lam = float(rng.uniform(0.5, 2.0))
        table = mo.steering_table_c64(pos.tolist(), K, lam)
        kind = trial % 3
        x = (rng.standard_normal((W, snaps, m)) + 1j * rng.standard_normal((W, snaps, m))) * (1.0 if kind else 1e-3)
        if kind == 1:  # plus sources on grid rows
            for w in range(W):
                for s in range(n):
                    a = table[int(rng.integers(0, K))].astype(np.complex128)
                    x[w] += 5.0 * a[None, :] * (rng.standard_normal((snaps, 1)) + 1j * rng.standard_normal((snaps, 1)))
        yield trial, m, n, snaps, K, table, x.reshape(W, snaps * m).astype(np.complex64)


def spectrum_at(spec, ref):
    return np.asarray(spec)[..., ref["spec_idx"]]


@pytest.mark.parametrize("path", helpers.golden_files(), ids=lambda p: p.split("/")[-1])
def test_reference_work_reproduces_the_golden_vectors(path):
    cfg, table, wins, x = golden_input(path)
    got = helpers.reference_result(FIXTURE, golden_key(path), x)
    K = cfg["resolution"]
    for i, w in enumerate(wins):
        filled = w["bins"] >= 0
        assert np.array_equal(angles_to_bins(got["angles"][i], K)[filled], w["bins"][filled])
        assert np.array_equal(got["angles"][i], w["angles"])  # float32 casts of k * 360 / K
        # float32 outputs: measured identical on every fixture; one float32 ulp of slack for another LAPACK build
        assert helpers.rel_err(got["levels"][i][filled], w["levels"][filled]) <= 1.2e-7
        assert helpers.rel_err(got["spectrum"][i], spectrum_at(w["spectrum"], got)) <= 1.2e-7


@pytest.mark.parametrize("base,over,W", SEEDED)
def test_oracles_follow_the_reference_on_seeded_windows(base, over, W):
    cfg, table, x = seeded_input(base, over, W)
    ref = helpers.reference_result(FIXTURE, helpers.case_key(base, over, W), x)
    c = co.work_batch(x, cfg["m"], cfg["n"], table, want_spectrum=True)
    assert np.array_equal(c["angles"], ref["angles"])
    assert helpers.rel_err(c["levels"], ref["levels"]) <= 1.2e-7  # float32 outputs, Jacobi vs LAPACK eigenvectors
    assert helpers.rel_err(spectrum_at(c["spectrum"], ref), ref["spectrum"]) <= 1.2e-7
    for w in range(W):
        py = mo.work(x[w], cfg["m"], cfg["n"], table)
        assert np.array_equal(py["angles"], ref["angles"][w])
        assert helpers.rel_err(py["levels"], ref["levels"][w]) <= 1.2e-7


def test_top_n_rule_on_the_mirror_symmetric_array():
    """x-axis ULA: P[k] == P[K - k] bit for bit on bit-equal table rows; the reference's strict '>' keeps the lower
    bin first and, for n = 2, reports the mirror bin second - the oracles' pick functions restate exactly that."""
    cfg, table, x = mirror_input()
    K = cfg["resolution"]
    ref = helpers.reference_result(FIXTURE, "mirror", x)
    c = co.work_batch(x, cfg["m"], 2, table)
    assert np.array_equal(c["angles"], ref["angles"])
    b = angles_to_bins(ref["angles"], K)
    mirrored = [w for w in range(10) if np.array_equal(table[b[w, 0]], table[(K - b[w, 0]) % K]) and b[w, 0] not in (0, K // 2)]
    assert mirrored, "no window with a bit-equal mirror row in this sample"
    for w in mirrored:
        assert b[w, 0] < K // 2 and b[w, 1] == K - b[w, 0]
        assert ref["levels"][w, 0] == ref["levels"][w, 1]


def test_random_small_shapes_against_the_reference_source():
    """sweep of small shapes: the C and numpy restatements must report the reference's angles exactly and its levels to
    float32 accuracy"""
    checked = 0
    for trial, m, n, snaps, K, table, x in random_small_shapes():
        # a rank-deficient R has exact eigenvalue ties: only compare where the spectrum is well conditioned
        if snaps < m:
            continue
        ref = helpers.reference_result(FIXTURE, "random_%d" % trial, x)
        if not (np.all(np.isfinite(ref["levels"])) and np.all(np.isfinite(ref["spectrum"]))):
            continue  # rank-deficient windows (snapshots < m - n) give 1/0: LAPACK- and Jacobi-dependent, skipped
        c = co.work_batch(x, m, n, table, want_spectrum=True)
        assert np.array_equal(c["angles"], ref["angles"]), (m, n, snaps, K)
        assert helpers.rel_err(c["levels"], ref["levels"]) <= 2e-6, (m, n, snaps, K)
        assert helpers.rel_err(spectrum_at(c["spectrum"], ref), ref["spectrum"]) <= 2e-6, (m, n, snaps, K)
        for w in range(x.shape[0]):
            py = mo.work(x[w], m, n, table)
            assert np.array_equal(py["angles"], ref["angles"][w]), (m, n, snaps, K)
        checked += 1
    assert checked >= 15
