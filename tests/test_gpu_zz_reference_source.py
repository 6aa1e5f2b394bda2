"""GPU (runs last): the CUDA path against the reference's OWN work() - the reference's lib/baz_music_doa.cc compiled
unmodified against stand-in GNU Radio / Armadillo headers (oracle/Makefile target `ref`, see tests/test_ref_shim.py).
What it returned on these inputs is stored in tests/golden/reference_source/gpu.npz
(tests/golden/make_reference_golden.py): angles and levels in full, the spectrum at the peak bins and a fixed sample of
the others.  The whole spectrum is checked against the C oracle on the same windows."""
import numpy as np
import pytest

from gr_baz_b200 import synth
from gr_baz_b200.music_doa import music_doa
from oracle import c_oracle as co

import helpers

pytestmark = pytest.mark.gpu

P_RTOL = 1e-5
FIXTURE = "gpu"

CASES = [
    (1, {}, 24), (1, {"n": 2}, 12), (2, {"snapshots": 1024}, 12), (4, {"snapshots": 512}, 10),
    (5, {"snapshots": 512, "resolution": 1800}, 8), (1, {"m": 6, "geometry": "uca", "n": 2}, 8),
    # the BASELINE shapes at FULL size (configs[1..4]): C2 4x4096x3600, C3 8x8192x7200, C4 8x4096x3600, C5 16x4096x3600 n=2
    (2, {}, 16), (3, {}, 8), (4, {}, 8), (5, {}, 8),
]


def case_input(base, over, W):
    cfg = synth.config(base, **over)
    return cfg, helpers.table_for(cfg), synth.gen_windows_numpy(cfg, 606 + base, 0, W)


@pytest.mark.parametrize("base,over,W", CASES)
def test_cuda_path_matches_the_reference_source(base, over, W):
    cfg, table, x = case_input(base, over, W)
    K, n = cfg["resolution"], cfg["n"]
    ref = helpers.reference_result(FIXTURE, helpers.case_key(base, over, W), x)
    blk = music_doa(cfg["m"], n, cfg["nsamples"], table.tolist(), K)
    ang = np.full((W, n), -7, np.float32)
    lvl = np.full((W, n), -7, np.float32)
    spec = np.zeros((W, K), np.float32)
    assert blk.work(W, [x], [ang, lvl, spec]) == W
    assert np.array_equal(ang, ref["angles"])  # = peak bins bit-exact (angle = (float)(k * 360 / K) is injective)
    assert helpers.rel_err(lvl, ref["levels"]) <= P_RTOL
    assert helpers.rel_err(spec[:, ref["spec_idx"]], ref["spectrum"]) <= P_RTOL
    assert helpers.rel_err(spec, co.work_batch(x, cfg["m"], n, table)["P"]) <= P_RTOL
    # peak-only call (the fused kernel for M = 4, n = 1)
    ang2 = np.zeros_like(ang)
    assert blk.work(W, [x], [ang2]) == W and np.array_equal(ang2, ref["angles"])
