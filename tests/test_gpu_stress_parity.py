"""GPU: every dispatcher route of the CUDA library on the adversarial windows of tests/stress_inputs.py, against the C
oracle and the reference's stored results, with proof of the route each call took.

A route is proved by the number of kernel launches the call made (music_b200.cu: the fused kernels are one launch; the
three-kernel path is covariance (cov4_tma / covN_tma: 1, cov_tile: 2, cov_generic: 1) + eigenvectors + scan, plus
top-n when n > 1 or in local-maximum mode, per sub-batch), by the fused M = 8 kernel's solver counters, and, for the fused
M = 4 kernel, by its trace words (MUSIC_B200_TRACE=1: word 15 = windows that took the all-fp64 fallback scan, word 19 =
rounds that needed the Jacobi solver).

Gates: bins and angles identical to the C oracle (a different bin only where the oracle's own P at the two bins agrees
to 1e-12, at most TIE_ALLOWANCE windows a call), levels and spectrum within 1e-5 of the oracle's P."""
import ctypes

import numpy as np
import pytest
import torch

from gr_baz_b200 import synth
from gr_baz_b200.music_doa import music_doa
from oracle import c_oracle as co
from oracle import music_oracle as mo

import helpers
import stress_inputs as si

pytestmark = pytest.mark.gpu

P_RTOL = 1e-5
TIE_ALLOWANCE = 2
SCAN_B = 8
MAX_SUB_M16_K36000 = 1352  # max_sub_windows(): 384 MiB / (16*16*2*8*2 + 16*8 + 36000*8) bytes, rounded down to SCAN_B
MAX_SUB_M16 = 48392  # the same without fp64 strengths in the workspace (d_P64 given): 384 MiB / (16*16*2*8*2 + 16*8), rounded down
DEV = torch.device("cuda:0")
ENV_KEYS = ("MUSIC_B200_FUSED", "MUSIC_B200_FUSED_SPEC", "MUSIC_B200_EIG", "MUSIC_B200_TRACE", "MUSIC_B200_MMA_FIN")


def make_block(monkeypatch, cfg, table, env=None):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    return music_doa(cfg["m"], cfg["n"], cfg["nsamples"], table.tolist(), cfg["resolution"])


def run_device(blk, cfg, x, spectrum=False, p64=False, internals=False):
    """x: (W, nsamples) complex64 (host).  One process_device() call; returns host outputs and the launch count."""
    W, n, K, M = x.shape[0], cfg["n"], cfg["resolution"], cfg["m"]
    d_in = torch.from_numpy(np.ascontiguousarray(x).view(np.float32)).to(DEV)
    d_ang = torch.full((W, n), -7.0, dtype=torch.float32, device=DEV)
    d_lvl = torch.full((W, n), -7.0, dtype=torch.float32, device=DEV)
    d_bins = torch.full((W, n), -7, dtype=torch.int32, device=DEV)
    d_spec = torch.full((W, K), -7.0, dtype=torch.float32, device=DEV) if spectrum else None
    d_P = torch.full((W, K), -7.0, dtype=torch.float64, device=DEV) if p64 else None
    d_R = torch.full((W, M, M, 2), -7.0, dtype=torch.float64, device=DEV) if internals else None
    d_ev = torch.full((W, M), -7.0, dtype=torch.float64, device=DEV) if internals else None
    ptr = lambda t: t.data_ptr() if t is not None else None
    torch.cuda.synchronize()
    l0 = blk.launch_count()
    blk.process_device(d_in.data_ptr(), W, d_ang.data_ptr(), d_lvl.data_ptr(), ptr(d_spec), d_bins.data_ptr(),
                       stream=torch.cuda.current_stream().cuda_stream, d_P64=ptr(d_P), d_R=ptr(d_R), d_eigvals=ptr(d_ev))
    torch.cuda.synchronize()
    out = dict(angles=d_ang.cpu().numpy(), levels=d_lvl.cpu().numpy(), bins=d_bins.cpu().numpy(), launches=blk.launch_count() - l0)
    if spectrum:
        out["spectrum"] = d_spec.cpu().numpy()
    if p64:
        out["P"] = d_P.cpu().numpy()
    if internals:
        R = d_R.cpu().numpy()
        out.update(R=R[..., 0] + 1j * R[..., 1], eigvals=d_ev.cpu().numpy())
    return out


def oracle(cfg, table, x, local=False):
    ref = co.work_batch(x, cfg["m"], cfg["n"], table, want_spectrum=False)
    if local:  # the opt-in local-maximum rule (oracle/music_oracle.py) on the C oracle's P
        for w in range(x.shape[0]):
            peaks = mo.pick_local_maxima(ref["P"][w], cfg["n"], cfg["resolution"])
            ref["bins"][w] = [p[2] for p in peaks]
            ref["angles"][w] = [p[0] for p in peaks]
            ref["levels"][w] = [p[1] for p in peaks]
    return ref


def assert_matches_oracle(got, ref, x, K):
    """bins / angles exact (up to TIE_ALLOWANCE oracle-decided ties), levels and spectrum to P_RTOL; non-finite windows
    give the untouched initial pair (angle 0, level 0, bin -1)"""
    bad = si.nonfinite_windows(x)
    assert np.all(got["bins"][bad] == -1) and np.all(got["angles"][bad] == 0) and np.all(got["levels"][bad] == 0)
    ties = 0
    for w in np.nonzero(~bad)[0]:
        gb, rb = got["bins"][w], ref["bins"][w]
        if not np.array_equal(gb, rb):
            P = ref["P"][w]
            for a, b in zip(gb, rb):
                assert a >= 0 and b >= 0 and abs(P[a] - P[b]) <= 1e-12 * abs(P[b]), (w, gb, rb)
            ties += 1
            continue
        assert np.array_equal(got["angles"][w], ref["angles"][w]), w
        ok = rb >= 0
        if ok.any():
            assert helpers.rel_err(got["levels"][w][ok], ref["levels"][w][ok]) <= P_RTOL, w
        assert np.all(got["levels"][w][~ok] == 0)
    assert ties <= TIE_ALLOWANCE, ties
    good = ~bad
    if "spectrum" in got and good.any():
        assert helpers.rel_err(got["spectrum"][good], ref["P"][good]) <= P_RTOL
    if "P" in got and good.any():
        assert helpers.rel_err(got["P"][good], ref["P"][good]) <= P_RTOL


def assert_matches_reference(got, key, x, K):
    """the reference's own work() on the fixture cases (tests/golden/reference_source/stress.npz)"""
    rec = helpers.reference_result("stress", key, x)
    good = ~si.nonfinite_windows(x)
    assert np.array_equal(got["angles"], rec["angles"])
    assert helpers.rel_err(got["levels"][good], rec["levels"][good]) <= P_RTOL
    if "spectrum" in got:
        assert helpers.rel_err(got["spectrum"][good][:, rec["spec_idx"]], rec["spectrum"][good]) <= P_RTOL


def same_outputs(a, b, rows=None):
    rows = slice(None) if rows is None else rows
    for k in ("bins", "angles", "levels", "spectrum", "P"):
        if k in a and k in b:
            assert np.array_equal(a[k][rows], b[k]), k


# ---- the route matrix -------------------------------------------------------------------------------------------------------
def unfused_launches(m, n, N, local=False, planar=False):
    """launches of one three-kernel sub-batch (music_b200.cu launch_cov / launch_eig_scan)"""
    if planar:
        cov = 1 if m <= 4 else 2
    elif m == 4:
        cov = 1                                   # cov4_tma_kernel
    elif m in (8, 16) and N >= 128 and N % (16 // m) == 0:
        cov = 1                                   # covN_tma_kernel<8|16>
    elif m % 4 == 0:
        cov = 1 if m == 4 else 2                  # cov_tile_kernel<false> + <true>
    else:
        cov = 1                                   # cov_generic_kernel
    return cov + 2 + (1 if (n > 1 or local) else 0)


# name: (env, spectrum port, case keys, launches per call (None: three-kernel count))
ROUTES = {
    "fused4_peaks": ({}, False, ["gap_m4", "coherent_m4", "highsnr_m4", "scaled_m4", "extreme_m4", "nonfinite_m4",
                                 "screen_36000", "screen_100000"], 1),
    "fused4_spectrum": ({}, True, ["gap_m4", "highsnr_m4", "scaled_m4", "extreme_m4", "nonfinite_m4", "screen_36000"], 1),
    "fused8": ({}, False, ["gap_m8", "coherent_m8", "highsnr_m8", "extreme_m8", "beams_m8"], 1),
    "unfused4": ({"MUSIC_B200_FUSED": "0"}, False, ["gap_m4", "highsnr_m4", "scaled_m4", "extreme_m4", "nonfinite_m4",
                                                   "screen_36000", "unequal_m4_n2", "route_m4_n3"], None),
    "unfused4_spectrum": ({"MUSIC_B200_FUSED_SPEC": "0"}, True, ["highsnr_m4", "nonfinite_m4", "unequal_m4_n2"], None),
    "unfused8": ({"MUSIC_B200_FUSED": "0"}, False, ["gap_m8", "coherent_m8", "highsnr_m8", "highsnr_m8_n2", "scaled_m8_n2",
                                                   "extreme_m8", "nonfinite_m8_n2", "unequal_m8_n3", "beams_m8"], None),
    "unfused8_spectrum": ({}, True, ["highsnr_m8", "nonfinite_m8_n2", "unequal_m8_n3"], None),
    "unfused16": ({}, False, ["route_m16_n2", "route_m16_n15"], None),
    "eig_coop12": ({}, False, ["route_m12_n2"], None),
    "generic": ({}, False, sorted(si.ROUTE_CASES_GENERIC), None),
}
ROUTE_ROWS = [(r, k) for r, (_, _, keys, _) in ROUTES.items() for k in keys]


@pytest.mark.parametrize("route,key", ROUTE_ROWS, ids=["%s-%s" % rk for rk in ROUTE_ROWS])
def test_route_matrix(monkeypatch, route, key):
    """every route on the windows that apply; measured max relative error of levels and spectrum <= 1e-8"""
    env, spectrum, _, launches = ROUTES[route]
    cfg, table, x = si.case(key)
    m, n, N, K = cfg["m"], cfg["n"], cfg["snapshots"], cfg["resolution"]
    blk = make_block(monkeypatch, cfg, table, env)
    got = run_device(blk, cfg, x, spectrum=spectrum)
    assert got["launches"] == (launches if launches is not None else unfused_launches(m, n, N)), got["launches"]
    ref = oracle(cfg, table, x)
    assert_matches_oracle(got, ref, x, K)
    if key in si.CASES:
        assert_matches_reference(got, key, x, K)
    bad = si.nonfinite_windows(x)
    if bad.any() or si.FAMILY.get(key) == "extreme":
        # neighbour independence: the batch without the non-finite (or extreme) windows gives the same bits elsewhere
        keep = ~bad if bad.any() else np.arange(x.shape[0]) % 2 == 0
        sub = run_device(blk, cfg, x[keep], spectrum=spectrum)
        same_outputs(got, sub, keep)
    if not bad.any() and si.FAMILY.get(key) != "extreme":
        # exact power-of-two scaling: R scales exactly, eigenvectors and P do not change by a bit
        for k in si.POW2_EXPONENTS:
            sc = run_device(blk, cfg, si.pow2_scaled(x, k), spectrum=spectrum)
            same_outputs(sc, {f: got[f] for f in ("bins", "levels", "spectrum") if f in got})
    blk.close()


@pytest.mark.parametrize("route", ["fused4", "fused4_spectrum", "fused8", "unfused4", "unfused8", "unfused16",
                                   "generic9", "generic15", "tile8", "eig_coop12", "local8"])
def test_small_windows_and_grids(monkeypatch, route):
    """W in {1, SCAN_B +- 1} and K in {1, 2, 3, FZ_BINS - 1, FZ_BINS, FZ_BINS + 1}: the fused kernel's table tiling and
    +inf padding rows, partial scan batches"""
    m, n, env, spectrum, N, launches = {
        "fused4": (4, 1, {}, False, 256, 1), "fused4_spectrum": (4, 1, {}, True, 256, 1),
        "fused8": (8, 1, {}, False, 256, 1), "unfused4": (4, 1, {"MUSIC_B200_FUSED": "0"}, False, 256, None),
        "unfused8": (8, 1, {"MUSIC_B200_FUSED": "0"}, False, 256, None), "unfused16": (16, 1, {}, False, 256, None),
        "generic9": (9, 4, {}, True, 100, None), "generic15": (15, 14, {}, False, 64, None),
        "tile8": (8, 1, {}, False, 127, None), "eig_coop12": (12, 2, {}, True, 64, None), "local8": (8, 7, {}, False, 256, None),
    }[route]
    local = route == "local8"
    for W, K in [(9, 1), (9, 2), (9, 3), (9, si.FZ_BINS - 1), (9, si.FZ_BINS), (1, si.FZ_BINS + 1), (SCAN_B - 1, si.FZ_BINS + 1),
                 (SCAN_B + 1, si.FZ_BINS + 1)]:
        cfg, table, x = si.route_case(m, n, snapshots=N, resolution=K, W=W, seed=K)
        blk = make_block(monkeypatch, cfg, table, env)
        if local:
            blk.set_peak_mode("local_maxima")
        got = run_device(blk, cfg, x, spectrum=spectrum)
        assert got["launches"] == (launches if launches is not None else unfused_launches(m, n, N, local)), (W, K, got["launches"])
        assert_matches_oracle(got, oracle(cfg, table, x, local), x, K)
        blk.close()


@pytest.mark.parametrize("m,N", [(8, 127), (8, 128), (8, 129), (8, 130), (8, 255), (8, 257), (16, 127), (16, 128), (16, 129),
                                 (16, 130), (16, 191), (16, 193)])
def test_covariance_edges(monkeypatch, m, N):
    """covN_tma_kernel<8|16> against cov_tile_kernel at N = 127 / 128 / 129 / 130 and one TMA stage (128 snapshots for
    M = 8, 64 for M = 16) +- 1 beyond the first: the route (launch count) and R itself (to 1e-12 of the oracle's)"""
    for n in (1, 2):
        cfg, table, x = si.route_case(m, n, snapshots=N, resolution=360, W=SCAN_B + 3, seed=N)
        blk = make_block(monkeypatch, cfg, table, {"MUSIC_B200_FUSED": "0"})
        got = run_device(blk, cfg, x, spectrum=False, internals=True)
        tma = N >= 128 and N % (16 // m) == 0
        assert got["launches"] == (1 if tma else 2) + 2 + (1 if n > 1 else 0)
        ref = oracle(cfg, table, x)
        assert_matches_oracle(got, ref, x, 360)
        for w in range(x.shape[0]):
            R = mo.covariance(x[w], m)
            assert np.max(np.abs(got["R"][w] - R)) <= 1e-12 * np.max(np.abs(R))
        blk.close()


def test_planar_routes(monkeypatch):
    """planar antenna streams: M = 4 on the fused kernel (one launch), M = 8 through cov_planar_kernel + eigenvectors + scan"""
    for key, launches in (("highsnr_m4", 1), ("highsnr_m8_n2", 2 + 2 + 1), ("scaled_m4", 1), ("nonfinite_m8_n2", 2 + 2 + 1)):
        cfg, table, x = si.case(key)
        m, N, W = cfg["m"], cfg["snapshots"], x.shape[0]
        streams = [np.ascontiguousarray(x.reshape(W, N, m)[:, :, r].reshape(-1)) for r in range(m)]
        blk = make_block(monkeypatch, cfg, table)
        ang = np.zeros((W, cfg["n"]), np.float32)
        lvl = np.zeros((W, cfg["n"]), np.float32)
        l0 = blk.launch_count()
        assert blk.work_planar(W, streams, [ang, lvl]) == W
        assert blk.launch_count() - l0 == launches
        got = dict(angles=ang, levels=lvl, bins=blk.last_bins().copy())
        assert_matches_oracle(got, oracle(cfg, table, x), x, cfg["resolution"])
        assert_matches_reference(got, key, x, cfg["resolution"])
        blk.close()


def _trace_words(blk, ctas=1):
    from gr_baz_b200 import _capi

    buf = (ctypes.c_longlong * (1024 * 32))()
    _capi.check(_capi.load().music_b200_debug_fused_trace(blk._h, buf, 1024), blk._h)
    return np.frombuffer(buf, np.int64).reshape(1024, 32)[:ctas]


def test_fused4_takes_the_jacobi_and_fallback_scan_routes(monkeypatch):
    """The traced fused M = 4 kernel: one window per call, the squaring solver hands exactly the windows with l2/l1
    above the squaring limit to the Jacobi solver; on the screen family (more than FZ_CMAX certain survivors on a
    non-flat spectrum, tensor-core passes to the end: MUSIC_B200_MMA_FIN=8) the all-fp64 fallback scan runs."""
    lim = si.squaring_limit()
    cfg, table, x = si.case("gap_m4")
    above = si.achieved_gap(cfg, x) > lim
    blk = make_block(monkeypatch, cfg, table, {"MUSIC_B200_TRACE": "1", "MUSIC_B200_MMA_FIN": "8"})
    ref = oracle(cfg, table, x)
    for w in range(x.shape[0]):
        got = run_device(blk, cfg, x[w:w + 1])
        assert got["launches"] == 1
        assert_matches_oracle(got, {k: ref[k][w:w + 1] for k in ("bins", "angles", "levels", "P")}, x[w:w + 1], cfg["resolution"])
        assert _trace_words(blk)[0, 19] == int(above[w]), (w, above[w])
    blk.close()
    for key in ("screen_36000", "screen_100000"):
        # tensor-core passes need several windows per CTA (otherwise every window goes to the fp64 drain workers): the
        # 6 windows, repeated
        cfg, table, x1 = si.case(key)
        reps = 2000
        x = np.tile(x1, (reps, 1))
        blk = make_block(monkeypatch, cfg, table, {"MUSIC_B200_TRACE": "1", "MUSIC_B200_MMA_FIN": "8"})
        got = run_device(blk, cfg, x)
        assert got["launches"] == 1
        tr = _trace_words(blk, 1024)
        assert tr[:, 15].sum() > 0 and tr[:, 7].sum() > 0, (key, tr[:, 7].sum(), tr[:, 15].sum())
        ref = oracle(cfg, table, x1)
        assert_matches_oracle({k: got[k][:6] for k in ("bins", "angles", "levels")}, ref, x1, cfg["resolution"])
        for k in ("bins", "angles", "levels"):
            assert np.array_equal(got[k].reshape(reps, 6, 1), np.broadcast_to(got[k][:6], (reps, 6, 1))), k
        blk.close()


def test_fused8_solver_split_on_the_gap_family(monkeypatch):
    """the fused M = 8 kernel solves the windows below the squaring limit by squaring and hands the others to Jacobi"""
    cfg, table, x = si.case("gap_m8")
    above = si.achieved_gap(cfg, x) > si.squaring_limit()
    blk = make_block(monkeypatch, cfg, table)
    s0 = blk.fused8_stats()
    got = run_device(blk, cfg, x)
    s1 = blk.fused8_stats()
    assert got["launches"] == 1
    assert (s1[0] - s0[0], s1[1] - s0[1]) == (int((~above).sum()), int(above.sum()))
    assert_matches_oracle(got, oracle(cfg, table, x), x, cfg["resolution"])
    blk.close()


@pytest.mark.parametrize("m", [4, 8])
def test_fused_and_unfused_agree_on_families(monkeypatch, m):
    """families 1-4: in Jacobi mode the fused kernel runs the unfused eigensolver's arithmetic - bins and levels
    bit-identical; in the default mode bins identical and levels to 1e-9"""
    keys = ["gap_m%d" % m, "coherent_m%d" % m, "highsnr_m%d" % m] + (["scaled_m4"] if m == 4 else [])
    for key in keys:
        cfg, table, x = si.case(key)
        outs = {}
        for name, env in (("unfused", {"MUSIC_B200_FUSED": "0"}), ("jacobi", {"MUSIC_B200_EIG": "jacobi"}), ("default", {})):
            blk = make_block(monkeypatch, cfg, table, env)
            outs[name] = run_device(blk, cfg, x)
            blk.close()
        assert outs["jacobi"]["launches"] == 1 and outs["default"]["launches"] == 1 and outs["unfused"]["launches"] == 3
        u = outs["unfused"]
        assert np.array_equal(outs["jacobi"]["bins"], u["bins"]) and np.array_equal(outs["jacobi"]["levels"], u["levels"]), key
        assert np.array_equal(outs["default"]["bins"], u["bins"]), key
        assert helpers.rel_err(outs["default"]["levels"], u["levels"]) <= 1e-9, key


def _check_every_window_against_single_runs(blk, cfg, table, x, got, spectrum, p64, internals, sample, windows=None):
    for w in (range(x.shape[0]) if windows is None else windows):
        one = run_device(blk, cfg, x[w:w + 1], spectrum=spectrum, p64=p64, internals=internals)
        for f in ("bins", "angles", "levels", "spectrum", "P", "R", "eigvals"):
            if f in one:
                assert np.array_equal(got[f][w:w + 1], one[f]), (w, f)
    ref = oracle(cfg, table, x[sample])
    assert_matches_oracle({k: v[sample] for k, v in got.items() if k != "launches"}, ref, x[sample], cfg["resolution"])


def test_sub_batches_with_every_output(monkeypatch):
    """M = 16, n = 2: MAX_SUB_M16 + 5 windows, two sub-batches through one workspace slot, with d_spec, d_P64, d_R and
    d_eigvals requested; windows on both sides of the boundary and a stride sample against single-window calls of the
    same handle, the sample against the oracle"""
    cfg = synth.config(5, snapshots=128, resolution=360)
    table = helpers.table_for(cfg)
    W = MAX_SUB_M16 + 5
    x = synth.gen_windows_numpy(cfg, 4049, 0, W)
    blk = make_block(monkeypatch, cfg, table)
    got = run_device(blk, cfg, x, spectrum=True, p64=True, internals=True)
    assert got["launches"] == 2 * unfused_launches(16, 2, 128)
    sample = np.unique(np.concatenate([np.arange(0, W, 4999), [MAX_SUB_M16 - 1, MAX_SUB_M16, MAX_SUB_M16 + 1, W - 1]]))
    _check_every_window_against_single_runs(blk, cfg, table, x, got, True, True, True, sample, windows=sample)
    for w in sample:
        R = mo.covariance(x[w], 16)
        assert np.max(np.abs(got["R"][w] - R)) <= 1e-12 * np.max(np.abs(R))
        assert np.max(np.abs(got["eigvals"][w] - np.linalg.eigvalsh(R))) <= 1e-11 * np.max(np.abs(R))
    blk.close()


def test_call_larger_than_one_workspace_slot(monkeypatch):
    """M = 16, n = 2, K = 36 000: more windows than max_sub_windows() lets one workspace slot hold (its fp64 strengths
    alone are K * 8 bytes a window): three sub-batches in one call"""
    cfg = synth.config(5, snapshots=128, resolution=36000)
    table = helpers.table_for(cfg)
    W = 2 * MAX_SUB_M16_K36000 + 5
    x = synth.gen_windows_numpy(cfg, 5036, 0, W)
    blk = make_block(monkeypatch, cfg, table)
    got = run_device(blk, cfg, x)
    assert got["launches"] == 3 * unfused_launches(16, 2, 128)
    sample = np.unique(np.concatenate([np.arange(0, W, 331), [MAX_SUB_M16_K36000 - 1, MAX_SUB_M16_K36000,
                                                             2 * MAX_SUB_M16_K36000, W - 1]]))
    _check_every_window_against_single_runs(blk, cfg, table, x, got, False, False, False, sample)
    blk.close()


@pytest.mark.parametrize("pinned", [False, True])
def test_host_path_over_several_chunks_with_the_spectrum_port(monkeypatch, pinned):
    """work() with the spectrum port and n = 2 over 3 full 32 MiB chunks plus a ragged tail (chunk = 32 MiB / (K * 4)
    windows = 233 at K = 36 000), pageable and pinned host memory: every window against the device path"""
    cfg = synth.config(1, n=2, snapshots=64, resolution=36000)
    table = helpers.table_for(cfg)
    chunk = (32 << 20) // (36000 * 4)
    W = 3 * chunk + 50
    x = synth.gen_windows_numpy(cfg, 777, 0, W)
    blk = make_block(monkeypatch, cfg, table)
    if pinned:
        xin = torch.from_numpy(x.view(np.float32)).pin_memory().numpy().view(np.complex64)
        ang = torch.zeros((W, 2), dtype=torch.float32).pin_memory().numpy()
        lvl = torch.zeros((W, 2), dtype=torch.float32).pin_memory().numpy()
        spec = torch.zeros((W, 36000), dtype=torch.float32).pin_memory().numpy()
    else:
        xin, ang, lvl, spec = x, np.zeros((W, 2), np.float32), np.zeros((W, 2), np.float32), np.zeros((W, 36000), np.float32)
    l0 = blk.launch_count()
    assert blk.work(W, [xin], [ang, lvl, spec]) == W
    assert blk.launch_count() - l0 == 4 * unfused_launches(4, 2, 64)  # 4 chunks
    host = dict(angles=ang, levels=lvl, spectrum=spec, bins=blk.last_bins().copy())
    dev = run_device(blk, cfg, x, spectrum=True)
    same_outputs(host, {k: dev[k] for k in ("bins", "angles", "levels", "spectrum")})
    sample = np.unique(np.concatenate([np.arange(0, W, 53), [chunk - 1, chunk, 2 * chunk, 3 * chunk, W - 1]]))
    assert_matches_oracle({k: v[sample] for k, v in host.items()}, oracle(cfg, table, x[sample]), x[sample], 36000)
    blk.close()
