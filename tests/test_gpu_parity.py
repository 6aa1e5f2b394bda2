"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against
the oracle on the same seeded inputs, against the committed golden fixtures, and - at
BASELINE.json's full sizes - through size-independent properties.

Gates (BASELINE.json north_star): peak-bin indices bit-exact; P(theta) <= 1e-5 relative."""
import os

import numpy as np
import pytest
import torch

from gr_baz_b200 import synth
from gr_baz_b200.music_doa import music_doa
from gr_baz_b200.music_doa_helper import music_doa_helper
from oracle import c_oracle as co
from oracle import music_oracle as mo

import helpers

pytestmark = pytest.mark.gpu

P_RTOL = 1e-5  # the north_star tolerance on P(theta)


def run_block(cfg, table, x, spectrum=True, device_path=False, want_internals=False):
    """x: (W, nsamples) complex64 host array.  Returns dict of host arrays."""
    W = x.shape[0]
    blk = music_doa(cfg["m"], cfg["n"], cfg["nsamples"], table.tolist(), cfg["resolution"])
    out = {}
    if not device_path:
        ang = np.full((W, cfg["n"]), -7, np.float32)
        lvl = np.full((W, cfg["n"]), -7, np.float32)
        outs = [ang, lvl]
        if spectrum:
            spec = np.zeros((W, cfg["resolution"]), np.float32)
            outs.append(spec)
            out["spectrum"] = spec
        assert blk.work(W, [x], outs) == W
        out.update(angles=ang, levels=lvl, bins=blk.last_bins().copy())
    else:
        dev = torch.device("cuda:0")
        d_in = torch.from_numpy(x.view(np.float32)).to(dev)
        d_ang = torch.empty((W, cfg["n"]), dtype=torch.float32, device=dev)
        d_lvl = torch.empty_like(d_ang)
        d_bins = torch.empty((W, cfg["n"]), dtype=torch.int32, device=dev)
        d_spec = torch.empty((W, cfg["resolution"]), dtype=torch.float32, device=dev) if spectrum else None
        d_P = torch.empty((W, cfg["resolution"]), dtype=torch.float64, device=dev) if want_internals else None
        d_R = torch.empty((W, cfg["m"], cfg["m"], 2), dtype=torch.float64, device=dev) if want_internals else None
        d_ev = torch.empty((W, cfg["m"]), dtype=torch.float64, device=dev) if want_internals else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        blk.process_device(ptr(d_in), W, ptr(d_ang), ptr(d_lvl), ptr(d_spec), ptr(d_bins),
                           stream=torch.cuda.current_stream().cuda_stream, d_P64=ptr(d_P), d_R=ptr(d_R), d_eigvals=ptr(d_ev))
        torch.cuda.synchronize()
        out.update(angles=d_ang.cpu().numpy(), levels=d_lvl.cpu().numpy(), bins=d_bins.cpu().numpy())
        if spectrum:
            out["spectrum"] = d_spec.cpu().numpy()
        if want_internals:
            R = d_R.cpu().numpy()
            out.update(P=d_P.cpu().numpy(), R=R[..., 0] + 1j * R[..., 1], eigvals=d_ev.cpu().numpy())
    out["launches"] = blk.launch_count()
    blk.close()
    return out


def assert_parity(got, ref, n, check_spectrum=True):
    assert np.array_equal(got["bins"], ref["bins"]), np.argwhere(got["bins"] != ref["bins"])[:5]
    assert np.array_equal(got["angles"], ref["angles"])
    valid = ref["bins"] >= 0
    assert helpers.rel_err(got["levels"][valid], ref["levels"][valid]) <= P_RTOL
    if check_spectrum and "spectrum" in got:
        assert helpers.rel_err(got["spectrum"], ref["P"]) <= P_RTOL
    if "P" in got:
        assert helpers.rel_err(got["P"], ref["P"]) <= P_RTOL


@pytest.mark.parametrize("path", helpers.golden_files(), ids=lambda p: os.path.basename(p)[:-4])
def test_golden_fixtures(path):
    cfg, seed, table, wins, _ = helpers.load_golden(path)
    x = np.stack([g["in"] for g in wins])
    ref = {k: np.stack([g[k] for g in wins]) for k in ("bins", "angles", "levels", "P", "R", "eigvals")}
    for device_path in (False, True):
        got = run_block(cfg, table, x, spectrum=True, device_path=device_path, want_internals=device_path)
        assert_parity(got, ref, cfg["n"])
        assert got["launches"] > 0
        if device_path:
            scale = np.max(np.abs(ref["R"]))
            assert np.max(np.abs(got["R"] - ref["R"])) <= 1e-12 * scale
            assert np.max(np.abs(got["eigvals"] - ref["eigvals"])) <= 1e-11 * scale
            assert helpers.rel_err(got["P"], ref["P"]) <= 1e-8  # far inside the 1e-5 gate


SEEDED = [
    # base cfg, overrides, windows
    (1, {}, 67),
    (1, dict(snr_db=0.0), 33),
    (1, dict(snr_db=40.0, geometry="ula_y"), 16),
    (1, dict(n=2, geometry="uca"), 16),
    (1, dict(n=3, geometry="uca"), 9),
    (1, dict(snapshots=128), 40),       # GRC default operating point
    (1, dict(snapshots=7), 8),          # fewer snapshots than lanes
    (1, dict(resolution=100), 8),       # K < one table tile
    (1, dict(resolution=777), 8),       # K not a multiple of the tile
    (2, {}, 24),
    (2, dict(snr_db=40.0), 8),
    (4, {}, 12),
    (4, dict(n=3), 5),
    (4, dict(n=5), 5),                  # n > M - n: direct noise-subspace form only
    (5, {}, 6),
    (5, dict(n=1, snapshots=512), 6),
    (1, dict(m=3, geometry="uca", n=1), 8),      # generic-M kernels
    (1, dict(m=5, geometry="uca", n=2), 8),
    (1, dict(m=6, geometry="uca", n=2, snapshots=200), 8),
    (1, dict(m=12, geometry="uca", n=2, snapshots=256), 6),
    (1, dict(m=2, geometry="ula_y", n=1, snapshots=256), 8),
]


@pytest.mark.parametrize("base,over,W", SEEDED, ids=lambda v: str(v).replace(" ", ""))
def test_seeded_batches_match_oracle(base, over, W):
    cfg = synth.config(base, **over)
    table = helpers.table_for(cfg)
    seed = synth.BASE_SEED + 100 + base
    x = synth.gen_windows_numpy(cfg, seed, 0, W)
    ref = co.work_batch(x, cfg["m"], cfg["n"], table, want_spectrum=False)
    got = run_block(cfg, table, x, spectrum=True, device_path=True, want_internals=True)
    assert_parity(got, ref, cfg["n"])
    got_h = run_block(cfg, table, x, spectrum=False, device_path=False)
    assert_parity(got_h, ref, cfg["n"])
    # numpy/LAPACK oracle on a couple of windows as well
    for w in (0, W - 1):
        r = mo.work(x[w], cfg["m"], cfg["n"], table)
        assert np.array_equal(got["bins"][w], r["bins"])
        assert helpers.rel_err(got["P"][w], r["P"]) <= P_RTOL


def test_edge_windows():
    cfg = synth.config(1)
    table = helpers.table_for(cfg)
    x = synth.gen_windows_numpy(cfg, 5, 0, 6)
    x[1] = 0  # all-zero window: R = 0, eigenvectors = identity
    x[3] *= np.float32(2.0 ** -60)  # tiny but normal
    x[4] *= np.float32(2.0 ** 40)   # large
    ref = co.work_batch(x, 4, 1, table)
    got = run_block(cfg, table, x, spectrum=True, device_path=True, want_internals=True)
    assert_parity(got, ref, 1)
    # NaN window: nothing is ever inserted (strict '>' is false for NaN): (0, 0), bin -1
    x[2, 17] = np.nan
    got = run_block(cfg, table, x, spectrum=False, device_path=False)
    assert got["bins"][2, 0] == -1 and got["angles"][2, 0] == 0.0 and got["levels"][2, 0] == 0.0
    assert np.array_equal(got["bins"][[0, 1, 3, 4, 5]], ref["bins"][[0, 1, 3, 4, 5]])
    # single window, single snapshot
    c1 = synth.config(1, snapshots=1)
    x1 = synth.gen_windows_numpy(c1, 9, 0, 1)
    assert_parity(run_block(c1, table, x1, device_path=True, want_internals=True), co.work_batch(x1, 4, 1, table), 1)


def test_mirror_ties_resolve_to_lower_bin():
    # x-axis ULA: P[k] == P[K-k] exactly; every bin must be computed by the same instruction
    # sequence so the tie is exact on the GPU too, and the lower bin must win.
    cfg = synth.config(1)
    table = helpers.table_for(cfg)
    x = synth.gen_windows_numpy(cfg, 4321, 0, 32)
    got = run_block(cfg, table, x, spectrum=True, device_path=True, want_internals=True)
    K = cfg["resolution"]
    k = np.arange(1, K // 2)
    k = k[np.all(table[k] == table[K - k], axis=1)]  # rows 90/270 and 120/240 differ in the c64 rounding of ~1e-16
    assert len(k) >= K // 2 - 4
    assert np.array_equal(got["P"][:, k], got["P"][:, K - k])
    ref = co.work_batch(x, cfg["m"], cfg["n"], table)
    assert np.array_equal(got["bins"], ref["bins"])
    # wherever the mirror rows are bit-equal the lower bin of the pair must have been reported
    tie = np.all(table[got["bins"][:, 0] % K] == table[(K - got["bins"][:, 0]) % K], axis=1)
    assert np.all(got["bins"][tie, 0] <= K // 2) and tie.sum() >= 28
    # the fused peak-only kernel (no spectrum/P64 requested) picks the same bins
    got2 = run_block(cfg, table, x, spectrum=False, device_path=True)
    assert np.array_equal(got2["bins"], got["bins"]) and helpers.rel_err(got2["levels"], got["levels"]) <= 1e-6


def test_optional_outputs_and_set_array_response():
    cfg = synth.config(1)
    x = synth.gen_windows_numpy(cfg, 77, 0, 10)
    hb = music_doa_helper(cfg["m"], cfg["n"], cfg["nsamples"], cfg["resolution"], synth.FREQUENCY, synth.SPACING,
                          cfg["antenna_array"], output_spectrum=False)
    ang = np.zeros((10, 1), np.float32)
    lvl = np.zeros((10, 1), np.float32)
    assert hb.work(10, [x], [ang, lvl]) == 10
    t0 = np.asarray(hb.array_response).astype(np.complex64)
    ref = co.work_batch(x, 4, 1, t0)
    assert np.array_equal(hb.impl.last_bins(), ref["bins"]) and np.array_equal(ang, ref["angles"])
    # only port 0 connected (the reference would dereference lvl == NULL here, :147-154)
    ang2 = np.zeros((10, 1), np.float32)
    assert hb.impl.work(10, [x], [ang2]) == 10 and np.array_equal(ang2, ang)
    # retune: new wavelength -> new table (python/music_doa_helper.py:100-103)
    hb.set_frequency(synth.FREQUENCY * 0.8)
    t1 = np.asarray(hb.array_response).astype(np.complex64)
    assert not np.array_equal(t0, t1)
    assert hb.work(10, [x], [ang, lvl]) == 10
    ref1 = co.work_batch(x, 4, 1, t1)
    assert np.array_equal(hb.impl.last_bins(), ref1["bins"]) and np.array_equal(ang, ref1["angles"])
    assert helpers.rel_err(lvl, ref1["levels"]) <= P_RTOL


def test_full_size_properties_config2():
    """BASELINE config 2 at full size (10k windows of M=4 x 4096 snapshots, 3600 angles) generated
    on the device: statelessness under permutation, exact invariance to power-of-two scaling,
    chunking independence, and oracle parity on a random subset."""
    cfg = synth.config(2)
    table = helpers.table_for(cfg)
    seed = synth.BASE_SEED + 2
    W = cfg["windows"]
    dev = torch.device("cuda:0")
    d_in = synth.gen_windows_torch(cfg, seed, 0, W, dev)
    blk = music_doa(cfg["m"], cfg["n"], cfg["nsamples"], table.tolist(), cfg["resolution"])

    def run(d_x, nw):
        a = torch.empty((nw, 1), dtype=torch.float32, device=dev)
        l = torch.empty((nw, 1), dtype=torch.float32, device=dev)
        b = torch.empty((nw, 1), dtype=torch.int32, device=dev)
        blk.process_device(d_x.data_ptr(), nw, a.data_ptr(), l.data_ptr(), None, b.data_ptr(),
                           stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return a.cpu().numpy(), l.cpu().numpy(), b.cpu().numpy()

    ang, lvl, bins = run(d_in, W)
    assert np.all((bins >= 0) & (bins < cfg["resolution"]))
    # mirror rule: the lower of (k, K-k) is reported
    tb = synth.true_bins(cfg, seed, 0, W)[:, 0]
    folded = np.minimum(tb, (cfg["resolution"] - tb) % cfg["resolution"])
    assert np.mean(np.abs(bins[:, 0] - folded) <= 2) > 0.95  # estimator sanity at 20 dB (endfire bins are coarse)
    # oracle parity on a random subset + first windows
    rng = np.random.default_rng(0)
    idx = np.unique(np.concatenate([np.arange(16), rng.integers(0, W, 48)]))
    x = d_in[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.complex64)
    ref = co.work_batch(x, cfg["m"], cfg["n"], table)
    assert np.array_equal(bins[idx], ref["bins"]) and np.array_equal(ang[idx], ref["angles"])
    assert helpers.rel_err(lvl[idx], ref["levels"]) <= P_RTOL
    # permutation: the block is stateless across windows
    perm = torch.randperm(W, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    a2, l2, b2 = run(d_in[perm].contiguous(), W)
    p = perm.cpu().numpy()
    assert np.array_equal(b2, bins[p]) and np.array_equal(l2, lvl[p])
    # power-of-two scaling: R scales exactly, rotations are identical -> P bit-identical
    a3, l3, b3 = run((d_in[:2048] * 4.0).contiguous(), 2048)
    assert np.array_equal(b3, bins[:2048]) and np.array_equal(l3, lvl[:2048])
    # a sub-range gives the same answers as the full batch (chunking independence)
    a4, l4, b4 = run(d_in[1234:1234 + 777], 777)
    assert np.array_equal(b4, bins[1234:2011]) and np.array_equal(l4, lvl[1234:2011])
    blk.close()


def test_full_size_single_windows_configs_3_and_5():
    for base, W in ((3, 3), (5, 4)):
        cfg = synth.config(base)
        table = helpers.table_for(cfg)
        x = synth.gen_windows_numpy(cfg, synth.BASE_SEED + base, 100, W)
        ref = co.work_batch(x, cfg["m"], cfg["n"], table)
        got = run_block(cfg, table, x, spectrum=True, device_path=True, want_internals=True)
        assert_parity(got, ref, cfg["n"])


@pytest.mark.parametrize("eig,mma_fin", [("power", "2"), ("jacobi", "2"), ("power", "-1"), ("jacobi", "8")])
def test_fused_kernel_matches_unfused_path_on_every_window(monkeypatch, eig, mma_fin):
    """Config 2 at full size through both device paths, for every one of the 10 000 windows, run after run
    (regression: partial final scan passes once skipped windows), and for window counts that leave ragged final
    passes / go through the drain workers only.
      eig = jacobi : the fused kernel runs the same Jacobi arithmetic as the unfused eig_kernel -> bins AND levels
                     must be BIT-identical to the unfused all-fp64 kernels (tensor-core screen + exact candidates,
                     drain workers, dynamic tickets change nothing);
      eig = power  : (default) principal eigenvector by squaring instead of Jacobi: an independent algorithm, so the
                     bins must be identical and the levels agree to 1e-9 (P is conditioned ~4000x, both are ~1e-12).
      mma_fin      : 2 = hand-over to the drain workers one covariance warp earlier than the default (3), -1 = fp64
                     drain workers only, 8 = tensor-core passes to the very end (the round-1 behaviour)."""
    cfg = synth.config(2)
    table = helpers.table_for(cfg)
    dev = torch.device("cuda:0")
    W = cfg["windows"]
    d_in = synth.gen_windows_torch(cfg, synth.BASE_SEED + 2, 0, W, dev)

    def run(fused, nw, reps):
        monkeypatch.setenv("MUSIC_B200_FUSED", "1" if fused else "0")
        monkeypatch.setenv("MUSIC_B200_EIG", eig)
        monkeypatch.setenv("MUSIC_B200_MMA_FIN", mma_fin)
        blk = music_doa(cfg["m"], cfg["n"], cfg["nsamples"], table.tolist(), cfg["resolution"])
        outs = []
        for _ in range(reps):
            a = torch.full((nw, 1), -7.0, dtype=torch.float32, device=dev)
            l = torch.full((nw, 1), -7.0, dtype=torch.float32, device=dev)
            b = torch.full((nw, 1), -7, dtype=torch.int32, device=dev)
            blk.process_device(d_in.data_ptr(), nw, a.data_ptr(), l.data_ptr(), None, b.data_ptr(),
                               stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            outs.append((a.cpu().numpy(), l.cpu().numpy(), b.cpu().numpy()))
        blk.close()
        return outs

    first = None
    for nw in (W, 1187, 9, 1):
        ref = run(False, nw, 1)[0]
        for got in run(True, nw, 3):
            assert np.array_equal(got[2], ref[2]) and np.array_equal(got[0], ref[0])
            if eig == "jacobi":
                assert np.array_equal(got[1], ref[1])
            else:
                assert helpers.rel_err(got[1], ref[1]) <= 1e-9
            if nw == W:  # run-to-run: the same launch gives the same bits whatever the ticket order was
                first = got if first is None else first
                assert np.array_equal(got[1], first[1])


def test_fused_kernel_degenerate_windows_take_the_jacobi_fallback():
    """Noise-only, all-zero, NaN and tiny windows inside a batch of ordinary ones: the principal-eigenvector solver must
    hand them to the Jacobi solver (no convergence / no trace to scale by) and the fused kernel must agree with the
    unfused path and the oracle on every window."""
    cfg = synth.config(2)
    table = helpers.table_for(cfg)
    W = 40
    x = synth.gen_windows_numpy(cfg, 99, 0, W)
    rng = np.random.default_rng(3)
    for w in (3, 11, 12, 30):  # noise only: eigenvalue ratios ~1.02
        x[w] = (rng.standard_normal(x.shape[1]) + 1j * rng.standard_normal(x.shape[1])).astype(np.complex64)
    x[5] = 0
    x[17] *= np.float32(2.0 ** -60)
    x[18] *= np.float32(2.0 ** 40)
    ref = co.work_batch(x, 4, 1, table)
    got = run_block(cfg, table, x, spectrum=False, device_path=True)
    assert_parity(got, ref, 1)
    x[7, 100] = np.nan
    got = run_block(cfg, table, x, spectrum=False, device_path=True)
    ok = np.arange(W) != 7
    assert got["bins"][7, 0] == -1 and got["angles"][7, 0] == 0.0 and got["levels"][7, 0] == 0.0
    assert np.array_equal(got["bins"][ok], ref["bins"][ok])


def test_fused_kernel_spectrum_port_matches_three_kernel_path(monkeypatch):
    """Port 2 connected (/root/reference/lib/baz_music_doa.cc:120-121) on the fused M = 4 kernel: every window goes through the
    fp64 drain workers, which write (float)P[k]; against the three-kernel path (bins and angles identical, spectrum and
    levels to 1e-9: different eigensolvers) and the oracle, with degenerate windows and window counts that leave partial groups."""
    cfg = synth.config(2)
    table = helpers.table_for(cfg)
    W = 333
    x = synth.gen_windows_numpy(cfg, 4242, 0, W)
    rng = np.random.default_rng(9)
    x[3] = (rng.standard_normal(x.shape[1]) + 1j * rng.standard_normal(x.shape[1])).astype(np.complex64)  # noise only
    x[5] = 0
    x[17] *= np.float32(2.0 ** -60)
    for nw in (W, 9, 1):
        monkeypatch.setenv("MUSIC_B200_FUSED_SPEC", "1")
        got = run_block(cfg, table, x[:nw], spectrum=True, device_path=True)
        monkeypatch.setenv("MUSIC_B200_FUSED_SPEC", "0")
        ref = run_block(cfg, table, x[:nw], spectrum=True, device_path=True)
        assert got["launches"] < ref["launches"]  # table preparation + ONE launch
        cmp = np.arange(nw) != 5  # (all-zero window: a flat spectrum whose argmax is decided by the last bit of either formula)
        assert np.array_equal(got["bins"][cmp], ref["bins"][cmp]) and np.array_equal(got["angles"][cmp], ref["angles"][cmp])
        ok = np.isfinite(ref["spectrum"]).all(axis=1)
        assert ok.sum() >= nw - 1
        assert helpers.rel_err(got["spectrum"][ok], ref["spectrum"][ok].astype(np.float64)) <= 1e-6  # float32 outputs
        assert helpers.rel_err(got["levels"][ok], ref["levels"][ok]) <= 1e-6
    monkeypatch.setenv("MUSIC_B200_FUSED_SPEC", "1")
    sub = x[:24]
    oracle = co.work_batch(sub, 4, 1, table, want_spectrum=True)
    got = run_block(cfg, table, sub, spectrum=True, device_path=True)
    okw = np.arange(24) != 5  # (the all-zero window has no defined eigenvectors)
    assert np.array_equal(got["bins"][okw], oracle["bins"][okw])
    assert helpers.rel_err(got["spectrum"][okw], oracle["P"][okw]) <= P_RTOL
    # a NaN window: untouched initial pair (angle 0, level 0, bin -1), NaN spectrum row, neighbours unaffected
    sub = sub.copy()
    sub[7, 100] = np.nan
    got = run_block(cfg, table, sub, spectrum=True, device_path=True)
    assert got["bins"][7, 0] == -1 and got["angles"][7, 0] == 0.0 and got["levels"][7, 0] == 0.0
    assert np.isnan(got["spectrum"][7]).all()
    keep = okw & (np.arange(24) != 7)
    assert np.array_equal(got["bins"][keep], oracle["bins"][keep])


@pytest.mark.parametrize("base,over", [(4, {}), (3, {"snapshots": 1000, "resolution": 777}), (4, {"snapshots": 130, "snr_db": 0.0})])
def test_fused_m8_kernel_matches_unfused_path_and_oracle(monkeypatch, base, over):
    """M = 8, n = 1, peak outputs: the fused persistent kernel (music_fused8.cuh) against the three-kernel path on every
    window (bins identical, levels to 1e-9: different eigensolvers), against the oracle on a subset, for window counts that
    leave partial scan batches, with degenerate windows (Jacobi fallback) mixed in, and bit-identical in Jacobi mode."""
    cfg = synth.config(base, **over)
    table = helpers.table_for(cfg)
    dev = torch.device("cuda:0")
    W = 2500
    d_in = synth.gen_windows_torch(cfg, synth.BASE_SEED + 40 + base, 0, W, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    for w in (7, 100, 1203):  # noise only: no dominant eigenvalue
        d_in[w] = torch.randn(d_in.shape[1], device=dev, generator=g)
    d_in[55] = 0
    d_in[56] *= 2.0 ** -50

    def run(fused, eig, nw):
        monkeypatch.setenv("MUSIC_B200_FUSED", "1" if fused else "0")
        monkeypatch.setenv("MUSIC_B200_EIG", eig)
        blk = music_doa(cfg["m"], cfg["n"], cfg["nsamples"], table.tolist(), cfg["resolution"])
        a = torch.full((nw, 1), -7.0, dtype=torch.float32, device=dev)
        l = torch.full((nw, 1), -7.0, dtype=torch.float32, device=dev)
        b = torch.full((nw, 1), -7, dtype=torch.int32, device=dev)
        for _ in range(2):
            blk.process_device(d_in.data_ptr(), nw, a.data_ptr(), l.data_ptr(), None, b.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        stats = blk.fused8_stats()
        launches = blk.launch_count()
        blk.close()
        return a.cpu().numpy(), l.cpu().numpy(), b.cpu().numpy(), stats, launches

    for nw in (W, 33, 5, 1):
        ref = run(False, "power", nw)
        got = run(True, "power", nw)
        assert got[4] == 1 + 2 and ref[4] > got[4]  # table preparation + ONE launch per call
        assert got[3][0] + got[3][1] == 2 * nw
        if nw == W:
            # the all-zero window must take the Jacobi fallback (no trace to scale by); noise-only windows may converge
            # by squaring (an eigenvalue ratio of 1.02 becomes 1.02^4096 after 12 squarings) or fall back
            assert 2 * 1 <= got[3][1] <= 2 * 12
        assert np.array_equal(got[2], ref[2]) and np.array_equal(got[0], ref[0])
        assert helpers.rel_err(got[1], ref[1]) <= 1e-9
        jac = run(True, "jacobi", nw)
        assert jac[3][0] == 0
        assert np.array_equal(jac[2], ref[2]) and np.array_equal(jac[1], ref[1])  # same Jacobi arithmetic: bit-identical
    idx = np.unique(np.concatenate([np.arange(12), [55, 56, 100, W - 1]]))
    x = d_in[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.complex64)
    oracle = co.work_batch(x, cfg["m"], cfg["n"], table)
    got = run(True, "power", W)
    assert np.array_equal(got[2][idx], oracle["bins"]) and np.array_equal(got[0][idx], oracle["angles"])
    assert helpers.rel_err(got[1][idx], oracle["levels"]) <= P_RTOL
