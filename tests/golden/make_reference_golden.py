#!/usr/bin/env python
"""Generates tests/golden/reference_source/ - what the reference itself returns on the inputs of the tests that compare
with it (tests/test_ref_shim.py, tests/test_gpu_zz_reference_source.py, tests/test_boundary_files.py).

  cpu.npz, gpu.npz, stress.npz
                    per test case: the angles and levels of the reference's own work() (oracle/_ref, built by
                    oracle/Makefile target `ref`), its spectrum at the peak bins plus a fixed sample of the others, and the
                    sha256 of the regenerated input (helpers.reference_record).
  surface.json      the signature of the reference's grc/baz_music_doa.xml and the declarations of its
                    lib/baz_music_doa.h that a drop-in must keep.

Run from the repo root, with the reference checkout at REFERENCE_DIR:
    python tests/golden/make_reference_golden.py REFERENCE_DIR
"""
import json
import os
import sys
import xml.etree.ElementTree as ET

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers  # noqa: E402
import stress_inputs  # noqa: E402
import test_boundary_files as tb  # noqa: E402
import test_gpu_zz_reference_source as tg  # noqa: E402
import test_ref_shim as tr  # noqa: E402
from oracle import ref_build  # noqa: E402


def record(d, key, x, cfg_m, n, K, table):
    res = ref_build.work_batch(x, cfg_m, n, table)
    for f, v in helpers.reference_record(x, K, res).items():
        d["%s/%s" % (key, f)] = v
    return res


def cpu_fixture():
    d = {}
    for path in helpers.golden_files():
        cfg, table, _, x = tr.golden_input(path)
        record(d, tr.golden_key(path), x, cfg["m"], cfg["n"], cfg["resolution"], table)
    for base, over, W in tr.SEEDED:
        cfg, table, x = tr.seeded_input(base, over, W)
        record(d, helpers.case_key(base, over, W), x, cfg["m"], cfg["n"], cfg["resolution"], table)
    cfg, table, x = tr.mirror_input()
    record(d, "mirror", x, cfg["m"], 2, cfg["resolution"], table)
    for trial, m, n, snaps, K, table, x in tr.random_small_shapes():
        if snaps < m:
            continue  # never compared
        res = record(d, "random_%d" % trial, x, m, n, K, table)
        kept = "random_%d/" % trial
        # the test decides finiteness from what is kept: it must decide as the whole result would
        assert (np.all(np.isfinite(res["levels"])) and np.all(np.isfinite(res["spectrum"]))) == \
            (np.all(np.isfinite(d[kept + "levels"])) and np.all(np.isfinite(d[kept + "spectrum"])))
    return d


def gpu_fixture():
    d = {}
    for base, over, W in tg.CASES:
        cfg, table, x = tg.case_input(base, over, W)
        record(d, helpers.case_key(base, over, W), x, cfg["m"], cfg["n"], cfg["resolution"], table)
    return d


def stress_fixture():
    d = {}
    for key in stress_inputs.CASES:
        cfg, table, x = stress_inputs.case(key)
        record(d, key, x, cfg["m"], cfg["n"], cfg["resolution"], table)
    return d


def surface(reference_dir):
    grc = ET.parse(os.path.join(reference_dir, "grc", "baz_music_doa.xml")).getroot()
    with open(os.path.join(reference_dir, "lib", "baz_music_doa.h")) as f:
        header = tb._norm(tb._decls(f.read()))
    decls = [tb._norm(s) for s in tb.CPP_SURFACE if tb._norm(s) in header]
    return {"grc_signature": json.loads(json.dumps(tb._sig(grc))), "cpp_declarations": decls}


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    if not ref_build.available():
        raise SystemExit("oracle/_ref is not built (oracle/Makefile target `ref`)")
    os.makedirs(helpers.REFERENCE_GOLDEN, exist_ok=True)
    for name, d in (("cpu", cpu_fixture()), ("gpu", gpu_fixture()), ("stress", stress_fixture())):
        np.savez_compressed(os.path.join(helpers.REFERENCE_GOLDEN, name + ".npz"), **d)
    with open(os.path.join(helpers.REFERENCE_GOLDEN, "surface.json"), "w") as f:
        json.dump(surface(sys.argv[1]), f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
