"""CPU tests (no GPU): pin the BA oracle restatement (oracle/ba_oracle.c) against the committed outputs
of the unmodified reference (tests/golden/ba_golden.npz, produced by tests/golden/make_ba_golden.py from
lib/sba-1.5 + lib/sfm-driver compiled in place) and, when oracle/_ref is built, against the reference
itself on a fresh scene (stored in tests/golden/reference_golden.npz).  Differences can only come from LAPACK's vs the
restatement's Cholesky rounding."""
import os

import numpy as np
import pytest

from bundler_sfm_b200 import bundle, synth

GOLD = os.path.join(os.path.dirname(__file__), "golden", "ba_golden.npz")
REF_GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz")


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def check(got, ref, nvis, what, ptol=1e-5):
    assert int(got["info"][5]) == int(ref["info"][5]), (what, got["info"][5], ref["info"][5])
    assert int(got["info"][6]) == int(ref["info"][6]), (what, got["info"][6], ref["info"][6])
    assert abs(np.sqrt(got["info"][1] / nvis) - np.sqrt(ref["info"][1] / nvis)) < 1e-9, what
    assert abs(got["info"][0] - ref["info"][0]) <= 1e-12 * abs(ref["info"][0]), what
    for key in ("R", "c", "f", "pts", "k"):
        assert rel(got[key], ref[key]) < ptol, (what, key, rel(got[key], ref[key]))


@pytest.mark.parametrize("name,kw", [
    ("syn10", {}),
    ("syn6nf", {"est_focal_length": 0, "undistort": 0}),
    ("syn8nd", {"est_focal_length": 1, "undistort": 0}),
    ("kermit", {}),
])
def test_port_matches_reference_golden(oracle, name, kw):
    g = np.load(GOLD)
    scene = {k: g[f"{name}_{k}"] for k in ("vmask", "projections", "R", "c", "f", "k", "pts")}
    ref = {k: g[f"{name}_ref_{k}"] for k in ("R", "c", "f", "k", "pts", "info")}
    got = oracle.run_sfm_port(scene, **kw)
    check(got, ref, scene["projections"].shape[0], name)


def test_port_matches_reference_golden_constraints(oracle):
    g = np.load(GOLD)
    scene = {k: g[f"kermitc_{k}"] for k in ("vmask", "projections", "R", "c", "f", "k", "pts")}
    ref = {k: g[f"kermitc_ref_{k}"] for k in ("R", "c", "f", "k", "pts", "info")}
    got = oracle.run_sfm_port(scene, use_constraints=1, constrained=g["kermitc_constrained"],
                              constraints=g["kermitc_constraints"], weights=g["kermitc_weights"])
    check(got, ref, scene["projections"].shape[0], "kermitc")


def test_port_vs_reference_fresh(oracle):
    """a scene outside ba_golden.npz, against the stored run_sfm results of the reference (tests/golden/make_reference_golden.py)"""
    g = np.load(REF_GOLD)
    scene = synth.ba_scene(7, 250, 4, seed=31)
    pc = np.zeros_like(scene["pts"]); pc[::5] = scene["gt_pts"][::5]
    for q, kw in enumerate(({}, {"ncons": 2}, dict(use_point_constraints=1, points_constraints=pc, point_constraint_weight=0.3))):
        got = oracle.run_sfm_port(scene, **kw)
        ref = {k: g[f"bafresh{q}_{k}"] for k in ("R", "c", "f", "k", "pts", "info")}
        check(got, ref, scene["projections"].shape[0], str(kw))


def test_golden_kermit_is_the_shipped_example():
    g = np.load(GOLD)
    # 11 images in the example, 9 of them registered in bundle.out; 2039 observations
    assert g["kermit_vmask"].shape[1] == 9 and g["kermit_projections"].shape[0] == 2039
    scene = {k: g[f"kermit_{k}"] for k in ("vmask", "projections", "R", "c", "f", "k", "pts")}
    sol = {k: g[f"kermit_ref_{k}"] for k in ("R", "c", "f", "k", "pts")}
    nvis = 2039
    # the reference's reported error is the reprojection error of the solution it returns
    assert abs(bundle.reprojection_rmse(scene, sol) - np.sqrt(g["kermit_ref_info"][1] / nvis)) < 1e-9
