"""Deterministic adversarial windows for the parity tests (numpy only, fixed seeds: the CPU and the GPU tests see the same
bytes).  Each family aims at one numerical mechanism of the CUDA kernels and returns (cfg, table, x), x being
(W, nsamples) complex64 in the block's item layout (x(r, c) = in[c * M + r]).

Signal model of the families (unlike gr_baz_b200/synth.py):
    X[c, r] = sum_s g_r sqrt(p_s) a_s[r] sym_s[c] + noise[c, r] (+ dc on one antenna)
with Walsh-Hadamard symbol sequences (rows of a Sylvester matrix, combined into unit-modulus complex symbols), so that
the sample cross-covariance of two sources is exactly zero for power-of-two snapshot counts and R has the structure the
family asks for.

The screen and squaring limits quoted below are derived in the functions that compute them (squaring_limit,
screen_survivors), from the constants of gr-baz_b200/csrc/music_eig4p.cuh and music_fused.cuh.
"""
import numpy as np

from gr_baz_b200 import synth
from oracle import music_oracle as mo

import helpers

EIGP_MAXSQ = 12             # music_eig4p.cuh: squarings of the principal-eigenvector solver (the extra one included)
RANK_ONE = 0.999999999      # its rank-one test ||A||_F^2 >= RANK_ONE tr(A)^2
FZ_CMAX = 256               # music_fused.cuh: exact candidates per window before the all-fp64 fallback scan
FZ_BINS = 448               # music_fused.cuh: table rows per tensor-core ring tile (16 * 7 scan warps * 4)
FZ_B = 2.0 ** -15           # music_fused.cuh: screen error bound relative to ||a||^2


def squaring_limit():
    """The eigenvalue ratio l2/l1 above which the squaring solver cannot converge.  Iteration it (0-based) squares once
    and tests A^(2^(it+1)); the test must pass by it = EIGP_MAXSQ - 2 so that one squaring is left.  With r = (l2/l1)^p
    the test reads (1 + r^2) / (1 + r)^2 >= RANK_ONE (further eigenvalues negligible), i.e. r <= r*."""
    lo, hi = 0.0, 1.0
    for _ in range(200):  # r*: largest r with (1 + r^2) >= RANK_ONE (1 + r)^2
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if 1.0 + mid * mid >= RANK_ONE * (1.0 + mid) ** 2 else (lo, mid)
    p = 2.0 ** (EIGP_MAXSQ - 1)
    return float(lo ** (1.0 / p))


def _hadamard(n):
    H = np.ones((1, 1))
    while H.shape[0] < n:
        H = np.block([[H, H], [H, -H]])
    return H


def _symbols(N, S, coherent=False):
    """(S, N) unit-modulus complex symbols from distinct Walsh-Hadamard rows (row 0, the constant, is skipped)"""
    H = _hadamard(max(2 * S + 2, N))[:, :N]
    rows = [(H[1] + 1j * H[2]) / np.sqrt(2.0)] * S if coherent else [(H[1 + 2 * s] + 1j * H[2 + 2 * s]) / np.sqrt(2.0) for s in range(S)]
    return np.stack(rows)


def _window(cfg, angles, powers, noise_power, rng, gains=None, noise_corr=0.0, dc=None, coherent=False):
    """One window (N, M) complex128 of the family model"""
    M, N = cfg["m"], cfg["snapshots"]
    a = synth.steering(cfg["antenna_array"], np.asarray(angles, np.float64))  # (S, M)
    sym = _symbols(N, len(angles), coherent)
    X = (sym.T * np.sqrt(np.asarray(powers, np.float64))) @ a  # (N, M)
    if noise_power > 0:
        z = (rng.standard_normal((N, M)) + 1j * rng.standard_normal((N, M))) * np.sqrt(noise_power / 2.0)
        if noise_corr:
            C = noise_corr ** np.abs(np.subtract.outer(np.arange(M), np.arange(M)))
            z = z @ np.linalg.cholesky(C).T
        X = X + z
    if gains is not None:
        X = X * np.asarray(gains)[None, :]
    if dc is not None:
        X[:, dc[0]] += dc[1]
    return X


def _pack(cfg, wins):
    """list of (N, M) complex128 -> (W, nsamples) complex64"""
    return np.stack([w.reshape(-1) for w in wins]).astype(np.complex64)


def _cfg(base, **over):
    cfg = synth.config(base, **over)
    return cfg, helpers.table_for(cfg)


def _bin_angle(cfg, k):
    return float(k) * 360.0 / cfg["resolution"]


# ---- 1 ------------------------------------------------------------------------------------------------------------------
GAP_TARGETS = (0.95, 0.965, 0.975, 0.982, 0.9915, 0.993, 0.996, 0.999)


def _orthogonal_partner(cfg, t1):
    """An angle t2 at least 30 degrees from t1 whose steering vector is orthogonal to a(t1) (a zero of the beam pattern)"""
    arr = cfg["antenna_array"]
    a1 = synth.steering(arr, t1)
    c = lambda t: np.abs(synth.steering(arr, t) @ np.conj(a1))
    grid = t1 + np.arange(30.0, 330.0, 0.01)
    t = float(grid[np.argmin(c(grid))])
    lo, hi = t - 0.01, t + 0.01
    for _ in range(100):  # |c| is V-shaped around a simple zero
        m1, m2 = lo + (hi - lo) / 3.0, hi - (hi - lo) / 3.0
        lo, hi = (lo, m2) if c(m1) < c(m2) else (m1, hi)
    return 0.5 * (lo + hi)


def eig_gap(m):
    """Eigenvalue gap around the squaring limit (principal eigenvector by repeated squaring, fused M = 4 / M = 8):
    two uncorrelated sources whose power ratio puts l2/l1 of R on both sides of squaring_limit()."""
    cfg, table = _cfg(2, snapshots=1024, resolution=720) if m == 4 else _cfg(4, snapshots=1024, resolution=720)
    rng = np.random.default_rng(101 + m)
    noise = 1e-5
    wins = []
    for i, rho in enumerate(GAP_TARGETS):
        t1 = 23.0 + 41.0 * i
        t2 = _orthogonal_partner(cfg, t1)  # a1^H a2 = 0: l2/l1 reaches 1 as p2 -> 1
        a = synth.steering(cfg["antenna_array"], np.array([t1, t2]))

        def ratio(p2):
            Rm = a[0][:, None] * a[0].conj() + p2 * a[1][:, None] * a[1].conj() + noise * np.eye(m)
            ev = np.linalg.eigvalsh(Rm)
            return ev[-2] / ev[-1]

        lo, hi = 0.0, 1.0
        for _ in range(60):  # ratio() is increasing in p2 on [0, 1]
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if ratio(mid) < rho else (lo, mid)
        wins.append(_window(cfg, [t1, t2], [1.0, lo], noise, rng))
    return cfg, table, _pack(cfg, wins)


def achieved_gap(cfg, x):
    """l2/l1 of each window's R, from the fp64 oracle's eigenvalues"""
    out = []
    for w in x:
        ev = np.linalg.eigvalsh(mo.covariance(w, cfg["m"]))
        out.append(ev[-2] / ev[-1])
    return np.array(out)


# ---- 2 ------------------------------------------------------------------------------------------------------------------
def unequal_sources(m, n):
    """Unequal sources, n = number of sources: 0 / -10 / -30 dB relative power at 40 dB SNR (noise subspace of a badly
    conditioned signal part)."""
    cfg, table = _cfg(2, m=m, n=n, snapshots=512, resolution=720, geometry="ula_x" if m == 4 else "uca")
    rng = np.random.default_rng(202 + 10 * m + n)
    powers = [1.0, 0.1, 0.001][:n]
    wins = []
    for i in range(6):
        angles = [17.0 + 53.0 * i + 71.0 * s + 0.37 * s for s in range(n)]
        wins.append(_window(cfg, angles, powers, 1e-4, rng))
    return cfg, table, _pack(cfg, wins)


def coherent_sources(m):
    """Two coherent sources (the same symbol sequence) with n = 1: R holds one merged rank-one signal term."""
    cfg, table = _cfg(2, m=m, n=1, snapshots=512, resolution=720, geometry="ula_x" if m == 4 else "uca")
    rng = np.random.default_rng(303 + m)
    wins = [_window(cfg, [31.0 + 47.0 * i, 121.0 + 29.0 * i], [1.0, 0.5], 1e-3, rng, coherent=True) for i in range(6)]
    return cfg, table, _pack(cfg, wins)


# ---- 3 ------------------------------------------------------------------------------------------------------------------
HIGH_SNR = (60.0, 80.0, None)  # None: noiseless
OFF_GRID = (0.5, 0.23, 1e-2, 1e-3, -1e-3)  # source offset from a grid row, in bins


def high_snr(m, n=1):
    """High SNR and rank deficiency: 60 dB, 80 dB and noiseless sources placed off-grid down to 1e-3 bin from a row
    (the noiseless R has m - n zero eigenvalues: Jacobi with zero off-diagonals, the certificate with l2 = 0, the
    2^-7 cancellation guard of the complement form at the peak)."""
    cfg, table = _cfg(2, m=m, n=n, snapshots=256, resolution=3600, geometry="ula_x" if m == 4 else "uca")
    rng = np.random.default_rng(404 + 10 * m + n)
    wins = []
    for i, snr in enumerate(HIGH_SNR):
        for j, off in enumerate(OFF_GRID):
            k0 = 137 + 331 * (3 * i + j)
            angles = [_bin_angle(cfg, k0 + off + 900 * s) for s in range(n)]
            wins.append(_window(cfg, angles, [1.0] * n, 0.0 if snr is None else 10.0 ** (-snr / 10.0), rng))
    return cfg, table, _pack(cfg, wins)


# ---- 4 ------------------------------------------------------------------------------------------------------------------
def badly_scaled(m, n=1):
    """Badly scaled R: per-antenna gains spread over 2^-10..2^10 (not powers of two), spatially correlated noise, a DC
    offset on one antenna (Jacobi stopping rules relative to ||R||_F)."""
    cfg, table = _cfg(2, m=m, n=n, snapshots=512, resolution=720, geometry="ula_x" if m == 4 else "uca")
    rng = np.random.default_rng(505 + 10 * m + n)
    wins = []
    for i in range(6):
        gains = 2.0 ** rng.uniform(-10.0, 10.0, m) * np.exp(1j * rng.uniform(0, 2 * np.pi, m))
        angles = [29.0 + 61.0 * i + 87.0 * s for s in range(n)]
        kind = i % 3
        wins.append(_window(cfg, angles, [1.0, 0.3][:n], 1e-3, rng, gains=gains if kind != 1 else None,
                            noise_corr=0.95 if kind == 1 else 0.0, dc=(m // 2, 0.4 + 0.2j) if kind == 2 else None))
    return cfg, table, _pack(cfg, wins)


# ---- 5 ------------------------------------------------------------------------------------------------------------------
def extreme_magnitudes(m):
    """Extreme magnitudes: ordinary windows scaled into the fp32 subnormal range (2^-140) and up to 2^120 (exact fp32 ->
    fp64 widening, fp64 products without overflow or underflow)."""
    cfg, table = _cfg(2, m=m, snapshots=512, resolution=720, geometry="ula_x" if m == 4 else "uca", snr_db=30.0)
    base = synth.gen_windows_numpy(cfg, 606 + m, 0, 6).astype(np.complex128)
    scales = (2.0 ** -140, 2.0 ** -133, 2.0 ** -126, 2.0 ** 100, 2.0 ** 117, 2.0 ** 120)
    return cfg, table, np.stack([b * s for b, s in zip(base, scales)]).astype(np.complex64)


POW2_EXPONENTS = (-100, -37, -1, 13, 60)


def pow2_scaled(x, k):
    """x * 2^k, exact for the ordinary windows used here (no fp32 subnormals or overflow for k in POW2_EXPONENTS)"""
    y = (x.astype(np.complex128) * 2.0 ** k).astype(np.complex64)
    assert np.array_equal((y.astype(np.complex128) * 2.0 ** -k).astype(np.complex64), x)
    return y


# ---- 6 ------------------------------------------------------------------------------------------------------------------
NONFINITE = (("+inf", np.inf), ("-inf", -np.inf), ("nan", np.nan), ("+inf imag", 1j * np.inf))


def non_finite(m, n=1):
    """Non-finite samples: one +Inf, -Inf or NaN in an otherwise ordinary window (even windows stay finite)."""
    cfg, table = _cfg(2, m=m, n=n, snapshots=256, resolution=720, geometry="ula_x" if m == 4 else "uca")
    x = synth.gen_windows_numpy(cfg, 707 + m, 0, 2 * len(NONFINITE))
    for i, (_, v) in enumerate(NONFINITE):
        pos = 37 * i + 5
        if np.iscomplexobj(v):
            x[2 * i + 1, pos] = np.complex64(complex(x[2 * i + 1, pos].real, np.inf))
        else:
            x[2 * i + 1, pos] = np.complex64(complex(v, x[2 * i + 1, pos].imag))
    return cfg, table, x


def nonfinite_windows(x):
    return ~np.all(np.isfinite(x), axis=1)


# ---- 7 ------------------------------------------------------------------------------------------------------------------
def screen_stress(K):
    """Screen stress: M = 4 ULA-x, K bins, 40-60 dB, sources near endfire where the spectrum is flat to fourth order, so
    that more than FZ_CMAX bins survive the 3xTF32 screen of a non-flat spectrum (the all-fp64 fallback scan)."""
    cfg, table = _cfg(2, snapshots=1024, resolution=K)
    rng = np.random.default_rng(808 + K % 1000)
    wins = []
    for i, (ang, snr) in enumerate(((0.7, 60.0), (179.3, 50.0), (2.9, 40.0), (181.1, 60.0), (90.4, 50.0), (355.2, 45.0))):
        wins.append(_window(cfg, [ang + 0.37 * 360.0 / K], [1.0], 10.0 ** (-snr / 10.0), rng))
    return cfg, table, _pack(cfg, wins)


def narrow_beams():
    """Narrow UCA-8 beams with near-equal adjacent bins: sources almost half-way between two rows at 60 dB."""
    cfg, table = _cfg(4, snapshots=512, resolution=7200)
    rng = np.random.default_rng(909)
    wins = [_window(cfg, [_bin_angle(cfg, 311 + 877 * i + off)], [1.0], 1e-6, rng)
            for i, off in enumerate((0.49, 0.499, 0.4999, 0.51, 0.501, 0.5001))]
    return cfg, table, _pack(cfg, wins)


def screen_survivors(table, e):
    """Bins that certainly pass the fused M = 4 screen for principal eigenvector e: with the exact d = ||a||^2 - |e^H a|^2
    and a screen error below FZ_B / 3 (tests/test_screen_bound.py), every bin with d <= d_min + (2 - 2/3) FZ_B ||a||^2
    is kept."""
    a = table.astype(np.complex128)
    na = np.sum(np.abs(a) ** 2, axis=1)
    d = na - np.abs(a @ np.conj(e)) ** 2
    return int(np.sum(d <= np.min(d) + (2.0 - 2.0 / 3.0) * FZ_B * na))


# ---- ordinary windows for the dispatcher routes ---------------------------------------------------------------------------
def route_case(m, n, snapshots=256, resolution=720, W=6, seed=0):
    """n sources from 0 to -12 dB at 30 dB SNR on a UCA, for the routes the families above do not reach: generic m,
    n = m - 1 (a one-dimensional noise subspace), covariance edges in N, small and odd K.  (Not a ULA: on an x-axis ULA
    the rows of 0 and 180 degrees differ only in the rounding of ~1e-16 imaginary parts, so K = 2 would be a tie.)"""
    cfg, table = _cfg(2, m=m, n=n, snapshots=snapshots, resolution=resolution, geometry="uca")
    rng = np.random.default_rng(1000 * m + 10 * n + seed)
    powers = list(10.0 ** (-np.linspace(0.0, 1.2, n)))
    wins = []
    for i in range(W):
        angles = list((11.0 + 29.0 * i + (360.0 / n) * np.arange(n) + rng.uniform(0.0, 7.0, n)) % 360.0)
        wins.append(_window(cfg, angles, powers, 1e-3, rng))
    return cfg, table, _pack(cfg, wins)


GENERIC_M = (7, 9, 11, 13, 15)
ROUTE_CASES = {"route_m%d_n%d" % (m, n): (lambda m=m, n=n: route_case(m, n)) for m in GENERIC_M for n in sorted({1, m // 2, m - 1})}
ROUTE_CASES_GENERIC = tuple(ROUTE_CASES)
ROUTE_CASES.update({"route_m8_n7": lambda: route_case(8, 7), "route_m12_n2": lambda: route_case(12, 2),
                    "route_m16_n2": lambda: route_case(16, 2), "route_m16_n15": lambda: route_case(16, 15),
                    "route_m4_n3": lambda: route_case(4, 3)})


# ---- registry -------------------------------------------------------------------------------------------------------------
CASES = {
    "gap_m4": lambda: eig_gap(4),
    "gap_m8": lambda: eig_gap(8),
    "unequal_m4_n2": lambda: unequal_sources(4, 2),
    "unequal_m8_n3": lambda: unequal_sources(8, 3),
    "coherent_m4": lambda: coherent_sources(4),
    "coherent_m8": lambda: coherent_sources(8),
    "highsnr_m4": lambda: high_snr(4),
    "highsnr_m8": lambda: high_snr(8),
    "highsnr_m8_n2": lambda: high_snr(8, 2),
    "scaled_m4": lambda: badly_scaled(4),
    "scaled_m8_n2": lambda: badly_scaled(8, 2),
    "extreme_m4": lambda: extreme_magnitudes(4),
    "extreme_m8": lambda: extreme_magnitudes(8),
    "nonfinite_m4": lambda: non_finite(4),
    "nonfinite_m8_n2": lambda: non_finite(8, 2),
    "screen_36000": lambda: screen_stress(36000),
    "screen_100000": lambda: screen_stress(100000),
    "beams_m8": narrow_beams,
}
FAMILY = {k: k.split("_")[0] for k in CASES}

_cache = {}


def case(key):
    if key not in _cache:
        _cache[key] = CASES[key]() if key in CASES else ROUTE_CASES[key]()
    return _cache[key]
