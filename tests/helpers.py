"""Shared helpers for the test-suite (oracle-side: allowed to import oracle/)."""
import glob
import hashlib
import os

import numpy as np

from gr_baz_b200 import synth
from oracle import music_oracle as mo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
# what the reference's own work() returned on the test inputs (tests/golden/make_reference_golden.py)
REFERENCE_GOLDEN = os.path.join(GOLDEN, "reference_source")
SPECTRUM_SAMPLE = 64  # spectrum bins kept per case besides the peak bins (keeps the fixtures small)

_table_cache = {}


def table_for(cfg):
    key = (cfg["geometry"], cfg["m"], cfg["resolution"])
    if key not in _table_cache:
        arr = mo.scaled_antenna_array(synth.SPACING, cfg["antenna_array"])
        _table_cache[key] = mo.steering_table_c64(arr, cfg["resolution"], synth.C_LIGHT / synth.FREQUENCY)
    return _table_cache[key]


def golden_files():
    return sorted(glob.glob(os.path.join(GOLDEN, "*.npz")))


def load_golden(path):
    """Returns (cfg, seed, table, list of per-window dicts incl. regenerated input)."""
    g = np.load(path)
    cfg = synth.config(int(g["base"]), m=int(g["m"]), n=int(g["n"]), snapshots=int(g["snapshots"]),
                       resolution=int(g["resolution"]), geometry=str(g["geometry"]), snr_db=float(g["snr_db"]))
    seed = int(g["seed"])
    table = g["table"] if "table" in g.files else table_for(cfg)
    wins = []
    for i, w in enumerate(g["windows"]):
        x = g["in_%d" % i] if ("in_%d" % i) in g.files else synth.gen_windows_numpy(cfg, seed, int(w), 1)[0]
        d = {k: g["%s_%d" % (k, i)] for k in ("R", "eigvals", "noise_projector", "P", "spectrum", "bins", "angles", "levels")}
        d["in"] = x
        d["in_sha256"] = str(g["in_sha256_%d" % i])
        d["w"] = int(w)
        wins.append(d)
    return cfg, seed, table, wins, str(g["table_sha256"])


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def sha256_of(x):
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


def case_key(base, over, W):
    return "c%d_%s_W%d" % (base, "_".join("%s%s" % kv for kv in sorted(over.items())), W)


def reference_record(x, K, res):
    """What a fixture keeps of one reference work_batch() result: angles and levels in full, the spectrum at the peak
    bins plus a fixed sample of the others (spec_idx), and the hash of the input it was computed from."""
    peaks = np.rint(np.asarray(res["angles"], np.float64) * K / 360.0).astype(np.int64) % K
    sample = np.random.default_rng(K).choice(K, min(K, SPECTRUM_SAMPLE), replace=False)
    idx = np.union1d(sample, peaks.ravel()).astype(np.int32)
    return {"angles": res["angles"], "levels": res["levels"], "spec_idx": idx, "spectrum": res["spectrum"][:, idx],
            "in_sha256": np.bytes_(sha256_of(x))}


_reference_cache = {}


def reference_result(fixture, key, x):
    """The stored reference result for case `key` of tests/golden/reference_source/<fixture>.npz; `x` must be the input
    it was recorded from."""
    if fixture not in _reference_cache:
        _reference_cache[fixture] = np.load(os.path.join(REFERENCE_GOLDEN, fixture + ".npz"))
    z = _reference_cache[fixture]
    rec = {f: z["%s/%s" % (key, f)] for f in ("angles", "levels", "spec_idx", "spectrum", "in_sha256")}
    assert sha256_of(x) == rec["in_sha256"].item().decode(), "input of case %s differs from the one the fixture was recorded on" % key
    return rec
