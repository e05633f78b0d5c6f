"""GPU parity tests of the BA path: every solve goes through the C ABI (bsfm_run_sfm in
libbsfm_b200.so) and is compared with (a) the committed outputs of the unmodified reference
(tests/golden/ba_golden.npz, made by tests/golden/make_ba_golden.py) and (b) the oracle run on the
GPU box (oracle/_ref when it was built, else the C restatement) on fresh synthetic scenes; where the C restatement has no
counterpart (motion-only solves, exported blocks, the dense solve alone) with the stored results of the reference on the same
inputs (tests/golden/reference_golden.npz, made by tests/golden/make_reference_golden.py).

Tolerances (BASELINE.json north_star): final reprojection RMSE within 1e-5 px; parameters within 1e-4
relative, measured per parameter group against the group's largest magnitude."""
import ctypes
import os

import numpy as np
import pytest

from bundler_sfm_b200 import bundle, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ba_golden.npz")
REF_GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RMSE_TOL = 1e-5
PARAM_TOL = 1e-4


def rel_group_err(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def check_solution(got, ref, nvis, what):
    r_gpu = np.sqrt(got["info"][1] / nvis)
    r_ref = np.sqrt(ref["info"][1] / nvis)
    assert abs(r_gpu - r_ref) <= RMSE_TOL, (what, r_gpu, r_ref)
    assert int(got["info"][5]) == int(ref["info"][5]), (what, "iterations", got["info"][5], ref["info"][5])
    assert int(got["info"][6]) == int(ref["info"][6]), (what, "stop reason", got["info"][6], ref["info"][6])
    for key in ("R", "c", "f", "pts"):
        err = rel_group_err(got[key], ref[key])
        assert err <= PARAM_TOL, (what, key, err)
    # distortion coefficients are O(1e-2): compare on the scale of the SBA parameter (k * k_scale=5) like the solver sees them
    assert np.max(np.abs(got["k"] - ref["k"])) * 5.0 <= PARAM_TOL * max(1.0, 5.0 * np.max(np.abs(ref["k"]))), (what, "k")
    assert abs(got["info"][0] - ref["info"][0]) <= 1e-9 * abs(ref["info"][0]), (what, "initial error")


def gold_scene(g, name):
    return {k: g[f"{name}_{k}"] for k in ("vmask", "projections", "R", "c", "f", "k", "pts")}


def gold_ref(g, name):
    return {k: g[f"{name}_ref_{k}"] for k in ("R", "c", "f", "k", "pts", "info")}


@pytest.mark.parametrize("name,kw", [
    ("syn10", {}),
    ("syn6nf", {"est_focal_length": 0, "undistort": 0}),
    ("syn8nd", {"est_focal_length": 1, "undistort": 0}),
    ("kermit", {}),
])
def test_golden_reference_outputs(name, kw):
    g = np.load(GOLD)
    scene = gold_scene(g, name)
    got = bundle.run_sfm(scene, **kw)
    check_solution(got, gold_ref(g, name), scene["projections"].shape[0], name)


def test_golden_with_camera_constraints():
    g = np.load(GOLD)
    scene = gold_scene(g, "kermitc")
    got = bundle.run_sfm(scene, use_constraints=1, constrained=g["kermitc_constrained"],
                         constraints=g["kermitc_constraints"], weights=g["kermitc_weights"])
    check_solution(got, gold_ref(g, "kermitc"), scene["projections"].shape[0], "kermitc")


def test_fresh_scene_vs_oracle(oracle):
    scene = synth.ba_scene(20, 2000, 5, seed=77)
    got = bundle.run_sfm(scene)
    ref = oracle.run_sfm_oracle(scene)
    check_solution(got, ref, scene["projections"].shape[0], "fresh20")
    # the solve must actually reduce the error and the reported error must match a numpy reprojection
    nvis = scene["projections"].shape[0]
    assert got["info"][1] < 0.05 * got["info"][0]
    assert abs(bundle.reprojection_rmse(scene, got) - np.sqrt(got["info"][1] / nvis)) < 1e-9


def test_point_constraints_vs_oracle(oracle):
    scene = synth.ba_scene(8, 300, 4, seed=9)
    pc = np.zeros_like(scene["pts"])
    pc[::7] = scene["gt_pts"][::7]
    kw = dict(use_point_constraints=1, points_constraints=pc, point_constraint_weight=0.5)
    got = bundle.run_sfm(scene, **kw)
    ref = oracle.run_sfm_oracle(scene, **kw)
    check_solution(got, ref, scene["projections"].shape[0], "ptcons")


def test_fixed_leading_cameras_vs_oracle(oracle):
    scene = synth.ba_scene(9, 400, 4, seed=12)
    got = bundle.run_sfm(scene, ncons=2)
    ref = oracle.run_sfm_oracle(scene, ncons=2)
    check_solution(got, ref, scene["projections"].shape[0], "mcon2")
    assert np.array_equal(got["c"][:2], scene["c"][:2])


def test_config2_vs_oracle(oracle):
    """BASELINE.json configs[1]: 50 cameras, 20k points, 100k observations"""
    scene = synth.ba_scene(50, 20000, 5, seed=1234)
    got = bundle.run_sfm(scene)
    ref = oracle.run_sfm_oracle(scene)
    check_solution(got, ref, 100000, "config2")


def test_analytic_jacobian_converges_to_same_optimum(monkeypatch):
    """fast mode: analytic Jacobian (not what the reference computes) must reach the same minimum to a
    looser tolerance -- it is a different LM trajectory, so only the optimum is compared"""
    scene = synth.ba_scene(12, 800, 4, seed=21)
    fd = bundle.run_sfm(scene)
    monkeypatch.setenv("BSFM_BA_JAC", "analytic")
    an = bundle.run_sfm(scene)
    nvis = scene["projections"].shape[0]
    assert abs(np.sqrt(an["info"][1] / nvis) - np.sqrt(fd["info"][1] / nvis)) < 2e-3


def test_unsupported_options_fail_loudly():
    import ctypes
    from bundler_sfm_b200._lib import load_library
    scene = synth.ba_scene(4, 60, 3, seed=1)
    lib = load_library()
    fn = lib.bsfm_run_sfm
    bundle.run_sfm(scene)   # binds argtypes
    vmask = np.ascontiguousarray(scene["vmask"], np.int8)
    cams = bundle.make_cameras(scene["R"], scene["c"], scene["f"], scene["k"])
    pts = scene["pts"].copy()
    proj = np.ascontiguousarray(scene["projections"])
    rc = fn(60, 4, 0, vmask.ctypes.data, proj.ctypes.data, 1, 0, 1, 1, ctypes.addressof(cams), pts.ctypes.data,
            0, 0, None, 0.0, 0, 1, 1e-12, None, None, None, None, None)   # optimize_for_fisheye = 1
    assert rc == -6 and b"fisheye" in lib.bsfm_last_error()
    S = np.zeros((36, 36))
    rc = fn(60, 4, 0, vmask.ctypes.data, proj.ctypes.data, 1, 0, 1, 1, ctypes.addressof(cams), pts.ctypes.data,
            0, 0, None, 0.0, 1, 0, 1e-12, None, S.ctypes.data, None, None, None)   # fix_points = 1 with an export buffer
    assert rc == -6 and b"fix_points" in lib.bsfm_last_error()


def test_config3_vs_reference_summary():
    """BASELINE.json configs[2]: 1000 cameras, 500k points, 3M observations against the stored summary of the
    reference run (tests/golden/ba_config3_ref.json, 835 s of CPU).  The reference stopped with reason 4 --
    its `pdp - 2 sqrt(p pdp) < -p` test (sba_levmar.c:1567) is a rounding knife-edge when eps4 = 0 -- so the
    iteration count may differ by one and the stop reason may be 4 or 8 (SURVEY.md H1); error and
    parameters must still agree."""
    import json
    ref = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ba_config3_ref.json")))
    scene = synth.ba_scene(1000, 500000, 6, seed=1234)
    got = bundle.run_sfm(scene)
    nvis = 3000000
    assert abs(np.sqrt(got["info"][1] / nvis) - np.sqrt(ref["info"][1] / nvis)) <= RMSE_TOL
    assert abs(int(got["info"][5]) - int(ref["info"][5])) <= 1
    assert int(got["info"][6]) in (4, 8)
    idx = np.array(ref["pt_idx"])
    assert rel_group_err(got["pts"][idx], np.array(ref["pts"])) <= PARAM_TOL
    assert rel_group_err(got["c"], np.array(ref["c"])) <= PARAM_TOL
    assert rel_group_err(got["f"], np.array(ref["f"])) <= PARAM_TOL
    assert rel_group_err(got["R"], np.array(ref["R"])) <= PARAM_TOL


def test_config3_equal_iteration_count_vs_reference():
    """SURVEY.md H1 / 8(d): the comparison "at equal iteration count", free of the eps4 = 0 knife-edge that decides where
    the full config-3 solve stops: both sides run exactly 4 LM iterations with Snavely's stop-8 rule disabled
    (itmax = 4, opts[5] = 0).  Reference summary: tests/golden/ba_config3_it4_ref.json (unmodified reference, 168 s)."""
    import json
    ref = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ba_config3_it4_ref.json")))
    scene = synth.ba_scene(1000, 500000, 6, seed=1234)
    n, m = scene["vmask"].shape
    nvis = scene["projections"].shape[0]
    p, cnp = bundle.pack_params(scene)
    vm = np.ascontiguousarray(scene["vmask"], np.int8)
    x = np.ascontiguousarray(scene["projections"])
    its, info = bundle.levmar_model(n, m, vm.ctypes.data, p.ctypes.data, x.ctypes.data, cnp, scene["R"], scene["f"], itmax=4, eps5=0.0)
    assert its == 4 and int(info[5]) == int(ref["info"][5]) == 4
    assert int(info[6]) == int(ref["info"][6]) == 3                        # stopped by itmax on both sides
    assert abs(info[0] - ref["info"][0]) <= 1e-9 * ref["info"][0]           # initial error
    assert abs(np.sqrt(info[1] / nvis) - np.sqrt(ref["info"][1] / nvis)) <= RMSE_TOL
    assert int(info[9]) == int(ref["info"][9])                             # same number of linear systems solved
    got = bundle.unpack_params(p, scene)
    idx = np.array(ref["pt_idx"])
    assert rel_group_err(got["pts"][idx], np.array(ref["pts"])) <= PARAM_TOL
    for key in ("c", "f", "R"):
        assert rel_group_err(got[key], np.array(ref[key])) <= PARAM_TOL, key


def test_mid_size_system_uses_blocked_path_vs_oracle(oracle):
    """200 cameras -> reduced system 1800 x 1800: exercises the large-system Cholesky path (diag/trsm kernels,
    DMMA trailing update, row-oriented back substitution) at a size the CPU reference finishes in seconds"""
    scene = synth.ba_scene(200, 6000, 6, seed=5)
    got = bundle.run_sfm(scene)
    ref = oracle.run_sfm_oracle(scene)
    check_solution(got, ref, scene["projections"].shape[0], "mid200")


def test_odd_pitch_system_vs_oracle(oracle):
    """cnp = 7 with 221 cameras -> reduced system dimension 1547 (> 1536: large path; odd row pitch: scalar access path)"""
    scene = synth.ba_scene(221, 4000, 5, seed=8)
    got = bundle.run_sfm(scene, undistort=0)
    ref = oracle.run_sfm_oracle(scene, undistort=0)
    check_solution(got, ref, scene["projections"].shape[0], "odd1547")


def test_multiwave_system_vs_oracle(oracle):
    """500 cameras -> reduced system 4500 x 4500: the per-step launches have more CTAs than the GPU holds at once
    (the case that exposed an intra-launch read/write race on the panel before the factor went out of place)"""
    scene = synth.ba_scene(500, 12000, 6, seed=15)
    got = bundle.run_sfm(scene)
    ref = oracle.run_sfm_oracle(scene)
    check_solution(got, ref, scene["projections"].shape[0], "multiwave500")


# ------------------------------------------------------------------------------------------------
# sba_Axb_Chol (sba_lapack.c:374-485): the dense SPD solve on its own, both Cholesky paths
# ------------------------------------------------------------------------------------------------
def _spd(n, seed, spread=2.0):
    rng = np.random.default_rng(seed)
    k = max(8, n // 4)
    G = rng.standard_normal((n, k))
    S = G @ G.T / k
    S += np.eye(n) * 1e-3 * np.trace(S) / n
    d = 10.0 ** rng.uniform(-spread, spread, n)
    S = S * d[:, None] * d[None, :]
    return (S + S.T) * 0.5


def _axb_chol(A, b):
    lib = bundle.load_library()
    fn = lib.bsfm_sba_Axb_Chol
    fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    fn.restype = ctypes.c_int
    x = np.zeros(A.shape[0])
    return fn(A.ctypes.data, b.ctypes.data, x.ctypes.data, A.shape[0], 0), x


@pytest.mark.parametrize("n", [9, 33, 64, 65, 255, 321, 450, 640, 641, 1547, 2100, 4000])
def test_axb_chol_vs_lapack(n):
    """single tile (<= 32), the one-launch dataflow path (<= 640, incl. partial last tiles and the two-tiles-per-CTA regime), the
    fused-step path (<= 1536) and the 256-column panel path with the tcgen05 int8-slice trailing update (> 1536), incl. an odd
    dimension and one that is not a multiple of 32: backward error at the level of LAPACK's, solution close to LAPACK's"""
    A = _spd(n, seed=n)
    xt = np.random.default_rng(1).standard_normal(n)
    b = A @ xt
    rc, x = _axb_chol(A, b)
    assert rc == 1
    xr = np.linalg.solve(A, b)
    nrm = np.linalg.norm(A, 'fro')
    res = np.linalg.norm(A @ x - b) / (nrm * np.linalg.norm(x))
    res_ref = np.linalg.norm(A @ xr - b) / (nrm * np.linalg.norm(xr))
    assert res <= max(10.0 * res_ref, 1e-14), (n, res, res_ref)
    # forward error bounded like LAPACK's own (the systems are ill-conditioned by construction: row scales 10^+-2)
    err, err_ref = np.linalg.norm(x - xt) / np.linalg.norm(xt), np.linalg.norm(xr - xt) / np.linalg.norm(xt)
    assert err <= max(20.0 * err_ref, 1e-10), (n, err, err_ref)


def test_axb_chol_vs_reference_routine():
    """the unmodified sba_Axb_Chol (dpotrf + dpotrs; its solution is stored in tests/golden/reference_golden.npz) on the same system"""
    g = np.load(REF_GOLD)
    n = 1800
    A = _spd(n, seed=3)
    b = A @ np.random.default_rng(2).standard_normal(n)
    rc, x = _axb_chol(A, b)
    xr = g["axb_x"]
    assert g["axb_rc"] == 1 and rc == 1
    assert np.linalg.norm(x - xr) / np.linalg.norm(xr) <= 1e-7


@pytest.mark.parametrize("n", [300, 2000])
def test_axb_chol_reports_indefinite_matrix(n):
    """the reference returns 0 when a leading minor is not positive definite (sba_lapack.c:439-442)"""
    A = _spd(n, seed=5)
    A[n // 2, n // 2] = -1.0
    rc, _ = _axb_chol(A, np.ones(n))
    assert rc == 0


def test_axb_chol_reports_indefinite_matrix_in_the_tail_of_a_large_system():
    """the last panels of the 256-column path are finished by the dataflow kernel: a bad pivot there is reported as well"""
    A = _spd(2000, seed=5)
    A[1900, 1900] = -1.0
    rc, _ = _axb_chol(A, np.ones(2000))
    assert rc == 0


def test_axb_chol_large_path_tail_hand_over_equals_panel_path():
    """n = 2600: with and without the dataflow hand-over of the last panels (BSFM_BA_CHOL_TAIL=0), each in a child process"""
    import subprocess
    import sys
    import tempfile
    code = ("import numpy as np, sys; sys.path.insert(0, %r); from tests.test_ba_gpu import _spd, _axb_chol; "
            "A = _spd(2600, 12); b = A @ np.random.default_rng(4).standard_normal(2600); rc, x = _axb_chol(A, b); "
            "assert rc == 1; np.save(sys.argv[1], x)") % ROOT
    with tempfile.TemporaryDirectory() as td:
        outs = []
        for tail in ("640", "0"):
            f = os.path.join(td, f"x{tail}.npy")
            subprocess.run([sys.executable, "-c", code, f], check=True, env=dict(os.environ, BSFM_BA_CHOL_TAIL=tail))
            outs.append(np.load(f))
    assert np.linalg.norm(outs[0] - outs[1]) / np.linalg.norm(outs[1]) <= 1e-7


def test_host_compressed_visibility_mask_equals_uploaded_mask():
    """large host-resident masks are scanned on the host and uploaded as CRS (ba_solver.cu: host_scan_vmask); forced here on a
    small scene (BSFM_BA_MASK_HOST_MIN=1, 3 scan threads) and compared bit for bit with the dense upload, in child processes"""
    import subprocess
    import sys
    import tempfile
    code = ("import numpy as np, sys; sys.path.insert(0, %r); from bundler_sfm_b200 import bundle, synth; "
            "sc = synth.ba_scene(12, 3000, 5, seed=3); out = bundle.run_sfm(sc); "
            "np.savez(sys.argv[1], info=out['info'], R=out['R'], c=out['c'], f=out['f'], k=out['k'], pts=out['pts'])") % ROOT
    with tempfile.TemporaryDirectory() as td:
        outs = []
        for host_min in ("1", str(1 << 40)):
            f = os.path.join(td, f"o{len(outs)}.npz")
            subprocess.run([sys.executable, "-c", code, f], check=True, env=dict(os.environ, BSFM_BA_MASK_HOST_MIN=host_min, BSFM_BA_MASK_THREADS="3"))
            outs.append(np.load(f))
    for key in ("info", "R", "c", "f", "k", "pts"):
        assert np.array_equal(outs[0][key], outs[1][key]), key


@pytest.mark.parametrize("n", [97, 450, 640])
def test_axb_chol_dataflow_equals_fused_step_path(n):
    """the cooperative dataflow factorisation (ba_chol_dataflow.cu) against the one-launch-per-32-columns path it replaces
    (BSFM_BA_CHOL_DATAFLOW=0), each in a child process"""
    import subprocess
    import sys
    import tempfile
    code = ("import numpy as np, sys; sys.path.insert(0, %r); from tests.test_ba_gpu import _spd, _axb_chol; "
            "n = int(sys.argv[2]); A = _spd(n, 21); b = A @ np.random.default_rng(4).standard_normal(n); rc, x = _axb_chol(A, b); "
            "assert rc == 1; np.save(sys.argv[1], x)") % ROOT
    with tempfile.TemporaryDirectory() as td:
        outs = []
        for df in ("1", "0"):
            f = os.path.join(td, f"x{df}.npy")
            subprocess.run([sys.executable, "-c", code, f, str(n)], check=True, env=dict(os.environ, BSFM_BA_CHOL_DATAFLOW=df))
            outs.append(np.load(f))
    assert np.linalg.norm(outs[0] - outs[1]) / np.linalg.norm(outs[1]) <= 1e-7


@pytest.mark.parametrize("where", [3, 200, 449])
def test_axb_chol_dataflow_reports_bad_pivot_anywhere(where):
    """a non-positive pivot in the first tile, in the middle and in the last (partial) tile of a 450 x 450 system"""
    A = _spd(450, seed=6)
    A[where, where] = -1.0
    rc, _ = _axb_chol(A, np.ones(450))
    assert rc == 0


def test_axb_chol_tensor_update_equals_dmma_update():
    """the tcgen05 int8-slice trailing update against the fp64 DMMA update (BSFM_BA_TC=0) in a child process"""
    import subprocess
    import sys
    code = ("import numpy as np, sys; sys.path.insert(0, %r); from tests.test_ba_gpu import _spd, _axb_chol; "
            "A = _spd(2600, 11); b = A @ np.random.default_rng(4).standard_normal(2600); rc, x = _axb_chol(A, b); "
            "assert rc == 1; np.save(sys.argv[1], x)") % ROOT
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        outs = []
        for tc in ("1", "0"):
            f = os.path.join(td, f"x{tc}.npy")
            subprocess.run([sys.executable, "-c", code, f], check=True, env=dict(os.environ, BSFM_BA_TC=tc))
            outs.append(np.load(f))
    assert np.linalg.norm(outs[0] - outs[1]) / np.linalg.norm(outs[1]) <= 1e-7


def test_export_of_U_V_W_S_vs_reference():
    """Vout/Sout/Uout/Wout (sba_levmar.c:1633-2026; Bundler asks for S in its first two-camera solve,
    src/Bundle.cpp:2150-2154): undamped blocks at the returned solution, against those the reference exported"""
    g = np.load(REF_GOLD)
    for m, n, L, keys in ((3, 80, 3, "S"), (6, 120, 3, "SUVW")):
        scene = synth.ba_scene(m, n, L, seed=40 + m)
        got = bundle.run_sfm(scene, export=keys)
        ref = {k: g[f"export{m}_{k}"] for k in ("R", "c", "f", "k", "pts", "info") + tuple(keys)}
        check_solution(got, ref, scene["projections"].shape[0], f"export{m}")
        for key in keys:
            scale = np.max(np.abs(ref[key]))
            # same gate as the parameters: the blocks are evaluated at solutions that agree to ~1e-7 and S = U - Y W^T cancels
            assert np.max(np.abs(got[key] - ref[key])) <= PARAM_TOL * scale, (m, key, np.max(np.abs(got[key] - ref[key])) / scale)
        assert np.allclose(got["S"], got["S"].T)


# ------------------------------------------------------------------------------------------------
# motion-only BA: run_sfm(fix_points = 1) -> sba_mot_levmar (sfm.c:843-849, sba_levmar.c:2090-2690)
# ------------------------------------------------------------------------------------------------
MOT_GOLD = os.path.join(os.path.dirname(__file__), "golden", "ba_mot_golden.npz")


def check_mot_solution(got, ref, scene, what):
    nvis = scene["projections"].shape[0]
    r_gpu = np.sqrt(got["info"][1] / nvis)
    r_ref = np.sqrt(ref["info"][1] / nvis)
    assert abs(r_gpu - r_ref) <= RMSE_TOL, (what, r_gpu, r_ref)
    # the reference stops these solves through stop rule 4 with eps4 = 0, i.e. when  pdp - 2 sqrt(p pdp) < -p  holds by
    # ROUNDING at convergence (sba_levmar.c:2596), or through rule 2: the iteration at which that happens is not a
    # property of the algorithm, so the count may differ by a few while the converged solution must agree
    assert abs(int(got["info"][5]) - int(ref["info"][5])) <= 3, (what, "iterations", got["info"][5], ref["info"][5])
    assert int(got["info"][6]) in (2, 4), (what, "stop reason", got["info"][6])
    assert abs(got["info"][0] - ref["info"][0]) <= 1e-9 * abs(ref["info"][0]), (what, "initial error")
    for key in ("R", "c", "f"):
        assert rel_group_err(got[key], ref[key]) <= PARAM_TOL, (what, key, rel_group_err(got[key], ref[key]))
    assert np.max(np.abs(got["k"] - ref["k"])) * 5.0 <= PARAM_TOL * max(1.0, 5.0 * np.max(np.abs(ref["k"]))), (what, "k")
    assert np.array_equal(got["pts"], scene["pts"]), (what, "points must stay fixed")


@pytest.mark.parametrize("name,kw", [("syn10", {}), ("syn6nf", {"est_focal_length": 0}), ("kermit", {})])
def test_motion_only_golden(name, kw):
    g = np.load(MOT_GOLD)
    scene = gold_scene(g, name)
    got = bundle.run_sfm(scene, fix_points=1, **kw)
    ref = {k: g[f"{name}_ref_{k}"] for k in ("R", "c", "f", "k", "info")}
    check_mot_solution(got, ref, scene, "mot_" + name)


def test_motion_only_golden_with_constraints():
    g = np.load(MOT_GOLD)
    scene = gold_scene(g, "syn10c")
    got = bundle.run_sfm(scene, fix_points=1, use_constraints=1, constrained=g["syn10c_constrained"],
                         constraints=g["syn10c_constraints"], weights=g["syn10c_weights"])
    ref = {k: g[f"syn10c_ref_{k}"] for k in ("R", "c", "f", "k", "info")}
    check_mot_solution(got, ref, scene, "mot_syn10c")


def test_motion_only_fresh_scene_vs_reference():
    """a larger motion-only solve against the stored result of the unmodified reference on the same scene"""
    g = np.load(REF_GOLD)
    scene = synth.ba_scene(40, 6000, 5, seed=31)
    got = bundle.run_sfm(scene, fix_points=1)
    ref = {k: g[f"motfresh_{k}"] for k in ("R", "c", "f", "k", "info")}
    check_mot_solution(got, ref, scene, "mot_fresh40")
    assert got["info"][1] < got["info"][0]
    assert got["info"][9] == 40 * (got["info"][7] - 1)     # one linear system per camera and function evaluation (:2513)
