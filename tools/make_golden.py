#!/usr/bin/env python
"""Regenerate the test vectors under tests/golden/ that stand in for files of the original project (Tom94/practical-path-guiding,
Mitsuba 0.5), so that the test suite runs from a clean checkout without it:

    python tools/make_golden.py <checkout of the original project>

Writes
  tests/golden/rough_transmittance_{beckmann,ggx}.npz   the nodes of mitsuba/data/microfacet/{beckmann,ggx}.dat that the rough-plastic
        materials of the tests interpolate (ppg_b200/rtrans.py: 4 eta x 4 alpha nodes per material, both eta halves, all theta samples);
        tests/conftest.py loads them with every other node NaN, so a material outside this set fails loudly instead of reading zeros.
  tests/golden/cbox/   cbox.xml and its meshes (scenes/cbox), the loader's input for scenes/cbox.npz.
  tests/golden/sky_model_rgb.npz   the RGB coefficient tables of mitsuba/src/emitters/sunsky/skymodeldata.h (ppg_b200/sunsky.py).
  tests/golden/reference_functions.npz   rows of the reference's outputs for the tests' seeded inputs (tests/reference_outputs.py), recorded by
        running those tests against oracle/_ref: build it first (`make -C oracle`, which needs the original project under REF_* paths).
  tests/golden/reference_digests.json   sha256 digests of the reference SD-tree's results in the same tests (trained trees are too large to store).
  tests/golden/reference_tree-02.sdt   the .sdt file the reference's own writer dumps in tests/test_oracle_sdtree.py::test_sdt_reader_reads_what_the_reference_writes.
"""
import os
import shutil
import sys

import pytest

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "practical-path-guiding_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from ppg_b200 import rtrans, sunsky  # noqa: E402
from common import load_rough_transmittance  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# (distribution, eta, alpha) of every rough plastic the tests reduce (tests/test_host_cpu.py, test_oracle_bsdf.py,
# test_device_source_on_host.py; the loader's defaults intIOR = polypropylene / extIOR = air, alpha 0.1, beckmann)
ROUGH_PLASTICS = [("beckmann", 1.49 / 1.000277, 0.1), ("beckmann", 1.49, 0.1), ("beckmann", 1.49, 0.4), ("beckmann", 1.5 / 1.000277, 0.1),
                  ("beckmann", 1.5 / 1.000277, 0.4), ("beckmann", 1.5, 0.02), ("beckmann", 1.5, 0.2), ("beckmann", 1.5, 0.4),
                  ("ggx", 1.5 / 1.000277, 0.2), ("ggx", 1.5, 0.02), ("ggx", 1.5, 0.025), ("ggx", 1.5, 0.04), ("ggx", 1.5, 0.05),
                  ("ggx", 1.5, 0.08), ("ggx", 1.5, 0.1), ("ggx", 1.5, 0.2), ("ggx", 1.5, 0.4)]


def _nodes(x, size):
    knot, _ = rtrans._weights(x, size)
    return [k for k in range(knot - 1, knot + 3) if 0 <= k < size]


def rough_transmittance(ref):
    data_dir = os.path.join(ref, "mitsuba", "data", "microfacet")
    for dist in ("beckmann", "ggx"):
        t = rtrans.load_table(dist, data_dir)
        keep = set()
        for d, eta, alpha in ROUGH_PLASTICS:
            if d != dist:
                continue
            alphas = _nodes(rtrans._warped_alpha(t, alpha), t["n_alpha"])
            for e in (np.float32(eta), np.float32(1.0 / eta)):          # external table (setEta(eta)) and internal diffuse (setEta(1 / eta))
                half = 0
                if e < 1:
                    half, e = t["n_eta"], np.float32(1) / e
                e = max(e, t["eta_min"])
                w = np.float32(np.power(np.float32((e - t["eta_min"]) / (t["eta_max"] - t["eta_min"])), np.float32(0.25)))
                keep |= {(half + k, a) for k in _nodes(w, t["n_eta"]) for a in alphas}
        idx = np.array(sorted(keep), np.int32)
        np.savez_compressed(os.path.join(GOLDEN, f"rough_transmittance_{dist}.npz"), index=idx,
                            trans=t["trans"][idx[:, 0], idx[:, 1]], diff=t["diff"][idx[:, 0], idx[:, 1]],
                            shape=np.array([t["n_eta"], t["n_alpha"], t["n_theta"]], np.int64),
                            ranges=np.array([t["eta_min"], t["eta_max"], t["alpha_min"], t["alpha_max"]], np.float32))
        full = {m: rtrans.reduce_for_material(d, eta, alpha, data_dir) for m, (d, eta, alpha) in enumerate(ROUGH_PLASTICS) if d == dist}
        rtrans._cache[dist] = load_rough_transmittance(dist)
        for m, (lut, fdr) in full.items():       # the sparse table reduces to the same bits
            lut2, fdr2 = rtrans.reduce_for_material(*ROUGH_PLASTICS[m])
            assert np.array_equal(lut, lut2) and fdr == fdr2, ROUGH_PLASTICS[m]
        print(f"rough_transmittance_{dist}.npz: {len(idx)} of {2 * t['n_eta'] * t['n_alpha']} (eta, alpha) nodes")


def cbox_scene(ref):
    src = os.path.join(ref, "scenes", "cbox")
    dst = os.path.join(GOLDEN, "cbox")
    os.makedirs(os.path.join(dst, "meshes"), exist_ok=True)
    shutil.copyfile(os.path.join(src, "cbox.xml"), os.path.join(dst, "cbox.xml"))
    for f in sorted(os.listdir(os.path.join(src, "meshes"))):
        shutil.copyfile(os.path.join(src, "meshes", f), os.path.join(dst, "meshes", f))


def sky_tables(ref):
    t = sunsky._sky_tables(os.path.join(ref, "mitsuba", "src", "emitters", "sunsky", "skymodeldata.h"))
    np.savez_compressed(os.path.join(GOLDEN, "sky_model_rgb.npz"), **t)


REFERENCE_TESTS = ["tests/test_oracle_bsdf.py::test_restated_microfacet_equals_the_reference_class",
                   "tests/test_oracle_bsdf.py::test_restated_helpers_equal_the_reference_functions",
                   "tests/test_oracle_bsdf.py::test_restated_triangle_test_and_spline_equal_the_reference",
                   "tests/test_oracle_bsdf.py::test_restated_discrete_distribution_equals_the_reference",
                   "tests/test_oracle_sunsky.py::test_sky_model_matches_the_reference_code",
                   "tests/test_oracle_sdtree.py::test_port_equals_verbatim_reference",
                   "tests/test_oracle_sdtree.py::test_restated_commit_equals_the_reference_vertex_commit",
                   "tests/test_oracle_sdtree.py::test_sdt_reader_reads_what_the_reference_writes"]


def reference_functions():
    assert os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libmicrofacet_ref.so")), "oracle/_ref is not built"
    import test_oracle_sdtree as T
    o, _ = T._run("ref", 2, 1, 0, iters=3, n=4000)
    assert o.dump(T.SDT_GOLDEN, T.SDT_CAM) == 0
    os.environ["PPG_RECORD_REFERENCE_OUTPUTS"] = "1"
    import reference_outputs
    reference_outputs.RECORD = "1"
    os.chdir(ROOT)
    assert pytest.main(["-q", "-p", "no:cacheprovider"] + REFERENCE_TESTS) == 0
    print(f"reference_functions.npz: {reference_outputs.save_recorded()} arrays")
    print(f"reference_digests.json: {reference_outputs.save_recorded_digests()} keys")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    rough_transmittance(sys.argv[1])
    cbox_scene(sys.argv[1])
    sky_tables(sys.argv[1])
    reference_functions()
