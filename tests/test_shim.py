"""The reference-facing link shims (shim/): run_sfm with the reference signature forwarding to the GPU
solver, and the UNMODIFIED reference KeyMatchFull main (src/KeyMatchFull.cpp) linked against the GPU
MatchKeys shim.  The CPU tests only check the artefacts exist and export the reference symbols; the GPU
tests run them."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from bundler_sfm_b200 import bundle, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "shim", "_build")
KM = os.path.join(BUILD, "KeyMatchFull_b200")
KMP = os.path.join(BUILD, "KeyMatchFull_b200_persistent")
KEYFILE = os.path.join(BUILD, "libkeyfile_b200.so")
SFMDRV = os.path.join(BUILD, "libsfmdrv_b200.so")
# what the unmodified reference returned on the inputs of these tests (tests/golden/make_reference_golden.py)
REF_GOLD = os.path.join(ROOT, "tests", "golden", "reference_golden.npz")


def test_sfmdrv_shim_exports_run_sfm():
    if not os.path.exists(SFMDRV):
        pytest.skip("shim/_build not built")
    lib = ctypes.CDLL(SFMDRV)
    assert hasattr(lib, "run_sfm")


def test_keymatchfull_shim_binary_links_reference_main():
    if not os.path.exists(KM):
        pytest.skip("shim/_build/KeyMatchFull_b200 not built (needs the reference sources at build time)")
    r = subprocess.run([KM], capture_output=True, text=True)
    assert "Usage:" in r.stdout and "<list.txt> <outfile> [window_radius]" in r.stdout   # KeyMatchFull.cpp:65


def _sha256(a):
    """digest under which tests/golden/make_reference_golden.py stores the descriptor lists the reference read"""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _read_with(fn, path):
    """call an `int f(const char *filename, unsigned char **keys[, keypt_t **info])` reader, return the descriptors"""
    buf = ctypes.POINTER(ctypes.c_ubyte)()
    fn.restype = ctypes.c_int
    n = fn(path.encode(), ctypes.byref(buf), None)
    if n <= 0:
        return n, None
    return n, np.ctypeslib.as_array(buf, shape=(n * 128,)).reshape(n, 128).copy()


def test_key_reader_equals_reference_readkeyfile(tmp_path):
    """shim/keyfile_b200.cpp against the stored results of the unmodified reference parser (src/keys2a.cpp:87-323) on the
    same files: plain file, gzip fallback, empty image, missing file, bad descriptor length."""
    if not os.path.exists(KEYFILE):
        pytest.skip("shim/_build not built")
    import gzip
    g = np.load(REF_GOLD)
    ref_n, ref_sha = g["keyfile_n"], g["keyfile_sha256"]
    ours = ctypes.CDLL(KEYFILE).bsfm_shim_read_key_file
    imgs = synth.sift_like_descriptors(3, [257, 1, 40], seed=5)
    for i, d in enumerate(imgs):
        p = str(tmp_path / f"a{i}.key")
        synth.write_key_file(p, d, seed=i)
        n1, k1 = _read_with(ours, p)
        assert ref_n[i] == n1 == d.shape[0] and _sha256(k1) == ref_sha[i] and np.array_equal(k1, d)
    # gzip fallback: only <name>.gz exists (keys2a.cpp:93-104)
    p = str(tmp_path / "z.key")
    synth.write_key_file(p, imgs[0], seed=9)
    with open(p, "rb") as f, gzip.open(p + ".gz", "wb") as gz:
        gz.write(f.read())
    os.remove(p)
    n1, k1 = _read_with(ours, p)
    assert ref_n[3] == n1 == 257 and _sha256(k1) == ref_sha[3]
    # empty image, missing file, wrong descriptor length: both return 0
    (tmp_path / "e.key").write_text("0 128\n")
    (tmp_path / "bad.key").write_text("1 64\n" + "1 2 3 4\n" + " ".join(["7"] * 64) + "\n")
    for q, name in enumerate(("e.key", "missing.key", "bad.key")):
        assert ref_n[4 + q] == 0
        assert _read_with(ours, str(tmp_path / name))[0] == 0


def test_persistent_keymatchfull_cli_usage():
    if not os.path.exists(KMP):
        pytest.skip("shim/_build/KeyMatchFull_b200_persistent not built")
    r = subprocess.run([KMP], capture_output=True, text=True)
    assert r.returncode != 0 and "Usage:" in r.stdout and "<list.txt> <outfile> [window_radius]" in r.stdout


def test_persistent_keymatchfull_cli_error_paths(tmp_path):
    """the argument / list-file errors of KeyMatchFull.cpp:25-56,64-90 are reported the same way, before any GPU work"""
    if not os.path.exists(KMP):
        pytest.skip("shim/_build/KeyMatchFull_b200_persistent not built")
    r = subprocess.run([KMP, str(tmp_path / "nope.txt"), str(tmp_path / "out.txt")], capture_output=True, text=True)
    assert r.returncode != 0 and "Error opening file" in r.stdout and "for reading." in r.stdout
    empty = tmp_path / "empty.txt"
    empty.write_text("\n   \n")
    r = subprocess.run([KMP, str(empty), str(tmp_path / "out.txt")], capture_output=True, text=True)
    assert r.returncode != 0 and "No input files found in" in r.stdout
    lst = tmp_path / "l.txt"
    lst.write_text("a.key\n")
    r = subprocess.run([KMP, str(lst), str(tmp_path / "no_such_dir" / "out.txt")], capture_output=True, text=True)
    assert r.returncode != 0 and "Could not open" in r.stdout and "for writing." in r.stdout


@pytest.mark.gpu
def test_persistent_keymatchfull_cli_writes_oracle_table(tmp_path, oracle):
    """SURVEY.md 8f row 2: KeyMatchFull's command line on the persistent matcher -> byte-identical matches.init.txt"""
    if not os.path.exists(KMP):
        pytest.skip("shim/_build/KeyMatchFull_b200_persistent not built")
    import gzip
    sizes = [700, 350, 0, 380, 300, 1200]
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=23)
    names = []
    for i, d in enumerate(imgs):
        p = tmp_path / f"img{i}.key"
        synth.write_key_file(str(p), d, seed=i)
        if i == 3:      # this one only exists gzipped
            with open(p, "rb") as f, gzip.open(str(p) + ".gz", "wb") as g:
                g.write(f.read())
            os.remove(p)
        names.append(str(p))
    lst = tmp_path / "list_keys.txt"
    lst.write_text("\n".join(names) + "\n\n")
    for window, extra in ((-1, []), (2, ["2"])):
        out = tmp_path / f"matches_{window}.txt"
        r = subprocess.run([KMP, str(lst), str(out)] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        want, _ = oracle.match_all_pairs_port(imgs, window, 0.6, 16)
        assert out.read_text() == want
        assert "[KeyMatchFull] Reading keys took" in r.stdout


@pytest.mark.gpu
def test_unmodified_keymatchfull_main_on_gpu_matches_oracle_table(tmp_path, oracle):
    if not os.path.exists(KM):
        pytest.skip("shim/_build/KeyMatchFull_b200 not built")
    sizes = [400, 350, 0, 380, 300]
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=17)
    names = []
    for i, d in enumerate(imgs):
        p = tmp_path / f"img{i}.key"
        synth.write_key_file(str(p), d, seed=i)
        names.append(str(p))
    lst = tmp_path / "list_keys.txt"
    lst.write_text("\n".join(names) + "\n")
    for window, extra in ((-1, []), (2, ["2"])):
        out = tmp_path / f"matches_{window}.txt"
        r = subprocess.run([KM, str(lst), str(out)] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        want, _ = oracle.match_all_pairs_port(imgs, window, 0.6, 16)
        assert out.read_text() == want


@pytest.mark.gpu
def test_run_sfm_through_reference_signature_shim(oracle):
    if not os.path.exists(SFMDRV):
        pytest.skip("shim/_build not built")
    lib = ctypes.CDLL(SFMDRV)
    fn = lib.run_sfm
    bundle._bind_run_sfm(fn)
    fn.restype = None
    scene = synth.ba_scene(8, 300, 4, seed=2)
    got = bundle.call_run_sfm(fn, scene)
    ref = oracle.run_sfm_oracle(scene)
    nvis = scene["projections"].shape[0]
    assert abs(bundle.reprojection_rmse(scene, got) - np.sqrt(ref["info"][1] / nvis)) <= 1e-5
    assert np.max(np.abs(got["pts"] - ref["pts"])) / np.max(np.abs(ref["pts"])) <= 1e-4


# ------------------------------------------------------------------------------------------------
# B2: sba_motstr_levmar / sba_mot_levmar with the reference signatures (shim/sba_b200.c), driven by a C program that is
# compiled against the reference's own sba.h (tests/c/sba_boundary_main.c, built by shim/Makefile)
# ------------------------------------------------------------------------------------------------
def _write_scene(path, scene, est_focal=1, undistort=1):
    vm = np.ascontiguousarray(scene["vmask"], np.int8)
    n, m = vm.shape
    proj = np.ascontiguousarray(scene["projections"], np.float64)
    with open(path, "wb") as f:
        f.write(np.array([n, m, proj.shape[0], est_focal, undistort], np.int32).tobytes())
        f.write(vm.tobytes()); f.write(proj.tobytes())
        cams = np.concatenate([np.asarray(scene["R"], float).reshape(m, 9), np.asarray(scene["c"], float), np.asarray(scene["f"], float)[:, None],
                               np.asarray(scene["k"], float)], axis=1)
        f.write(np.ascontiguousarray(cams).tobytes())
        f.write(np.ascontiguousarray(scene["pts"], np.float64).tobytes())


def _read_result(path, scene, cnp):
    raw = open(path, "rb").read()
    rc = int(np.frombuffer(raw[:4], np.int32)[0])
    info = np.frombuffer(raw[4:84], np.float64).copy()
    p = np.frombuffer(raw[84:], np.float64).copy()
    return rc, info, p


def _gold_ref(prefix, keys=("R", "c", "f", "k", "pts", "info")):
    g = np.load(REF_GOLD)
    return {k: g[f"{prefix}_{k}"] for k in keys}


@pytest.mark.gpu
def test_sba_motstr_levmar_reference_signature_program(tmp_path):
    from bundler_sfm_b200 import bundle
    exe = os.path.join(BUILD, "sba_boundary_test")
    if not os.path.exists(exe):
        pytest.skip("shim/_build/sba_boundary_test not built")
    scene = synth.ba_scene(12, 700, 4, seed=77)
    nvis = scene["projections"].shape[0]
    _write_scene(tmp_path / "scene.bin", scene)
    r = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "res.bin")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rc, info, p = _read_result(tmp_path / "res.bin", scene, 9)
    ref = _gold_ref("motstr")                # run_sfm of the unmodified reference on this scene
    assert rc == int(ref["info"][5]) == int(info[5])                    # returns the iteration count like the reference
    assert int(info[6]) == int(ref["info"][6])
    assert abs(np.sqrt(info[1] / nvis) - np.sqrt(ref["info"][1] / nvis)) <= 1e-5
    assert info[7] == ref["info"][7] and info[8] == ref["info"][8]      # simple driver scales nfev / njev by nvis (sba_levmar_wrap.c:684-695)
    got = bundle.unpack_params(p, scene)
    for key in ("R", "c", "f", "pts"):       # the parameter gate of tests/test_ba_gpu.py (relative to the group's scale)
        err = float(np.max(np.abs(got[key] - ref[key])) / np.max(np.abs(ref[key])))
        assert err <= 1e-4, (key, err)
    # a foreign projection callback is refused loudly with SBA_ERROR (no CPU fallback)
    r = subprocess.run([exe, "foreign"], capture_output=True, text=True)
    assert r.returncode == 0 and "foreign rc=-1" in r.stdout and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_sba_mot_levmar_reference_signature_program(tmp_path):
    exe = os.path.join(BUILD, "sba_boundary_test")
    if not os.path.exists(exe):
        pytest.skip("shim/_build/sba_boundary_test not built")
    from bundler_sfm_b200 import bundle
    scene = synth.ba_scene(10, 500, 4, seed=78)
    nvis = scene["projections"].shape[0]
    _write_scene(tmp_path / "scene.bin", scene)
    r = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "res.bin"), "mot"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rc, info, p = _read_result(tmp_path / "res.bin", scene, 9)
    ref = _gold_ref("mot", ("R", "c", "f", "k", "info"))      # run_sfm(fix_points = 1) of the unmodified reference
    assert abs(rc - int(ref["info"][5])) <= 3 and int(info[6]) in (2, 4)     # eps4 = 0 knife-edge, see test_ba_gpu.check_mot_solution
    assert abs(np.sqrt(info[1] / nvis) - np.sqrt(ref["info"][1] / nvis)) <= 1e-5
    got = bundle.unpack_params(p, scene)
    assert np.array_equal(got["pts"], np.asarray(scene["pts"], float))          # points untouched
    for key in ("c", "f"):
        assert float(np.max(np.abs(got[key] - ref[key])) / np.max(np.abs(ref[key]))) <= 1e-4, key


# ------------------------------------------------------------------------------------------------
# (f)4: MatchKeys(std::vector<KeypointWithDesc>...) of src/keys.cpp (bundler --add_images) -> GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_keys_cpp_matchkeys_overload_equals_reference_exhaustive(oracle):
    """shim/keys_b200.cpp (compiled against the reference's keys.h) against the unmodified MatchKeysExhaustive, for the two
    calls BundleRegisterImage makes (registered / 0.75 and unregistered / 1.0, Bundle.cpp:3812-3820) and more"""
    so = os.path.join(BUILD, "libkeys_b200.so")
    if not os.path.exists(so) or oracle.ref_keys() is None:
        pytest.skip("needs shim/_build/libkeys_b200.so and oracle/_ref/libref_keys.so")
    bundle.load_library()
    shim = ctypes.CDLL(so).shim_keys_match
    shim.argtypes = oracle.ref_keys().ref_keys_match.argtypes
    shim.restype = ctypes.c_int
    imgs = synth.sift_like_descriptors(3, [1800, 2300, 1], seed=12)
    extra = np.where(np.random.default_rng(4).random(2300) < 0.5, 7, -1).astype(np.int32)
    for reg, ratio in ((True, 0.75), (False, 1.0), (False, 0.6), (True, 0.95)):
        want = oracle.keys_match_ref(imgs[0], imgs[1], extra, reg, ratio, exhaustive=True)
        for exhaustive in (True, False):      # both names are exact on the GPU
            got = oracle.keys_match_ref(imgs[0], imgs[1], extra, reg, ratio, exhaustive=exhaustive, fn=shim)
            assert np.array_equal(got, want), (reg, ratio, exhaustive)
        assert want.shape[0] > 0
    # a database of one key aborts the reference (ANN: "Requesting more near neighbors than data points"); here d1 = INT_MAX
    # (ANN_DIST_INF) and every query matches it, like MatchKeys of keys2a.cpp does.  An empty registered set gives no match.
    assert oracle.keys_match_ref(imgs[0][:50], imgs[2], None, False, 0.75, fn=shim).shape[0] == 50
    none = np.full(2300, -1, np.int32)
    assert oracle.keys_match_ref(imgs[0][:50], imgs[1], none, True, 0.75, fn=shim).shape[0] == 0


@pytest.mark.gpu
def test_keys_cpp_test_on_real_sift_kermit_golden():
    g = np.load(os.path.join(ROOT, "tests", "golden", "kermit_match_golden.npz"))
    lib = bundle.load_library()
    fn = lib.bsfm_match_pair_test
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    fn.restype = ctypes.c_int
    for (a, b) in ((0, 1), (3, 7), (10, 9)):
        k1, k2 = np.ascontiguousarray(g[f"desc{a}"]), np.ascontiguousarray(g[f"desc{b}"])
        out = np.zeros((k1.shape[0], 2), np.int32)
        n = fn(k1.ctypes.data, k1.shape[0], k2.ctypes.data, k2.shape[0], 0.75, 1, out.ctypes.data, k1.shape[0])
        assert np.array_equal(out[:n], g[f"keys_{a}_{b}"]), (a, b)


@pytest.mark.gpu
def test_match_pair_test_modes_vs_port(oracle):
    lib = bundle.load_library()
    fn = lib.bsfm_match_pair_test
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    fn.restype = ctypes.c_int
    imgs = synth.sift_like_descriptors(2, [900, 1100], seed=13)
    for mode in (0, 1):
        for ratio in (0.6, 0.9, 1.0):
            out = np.zeros((900, 2), np.int32)
            n = fn(imgs[0].ctypes.data, 900, imgs[1].ctypes.data, 1100, ratio, mode, out.ctypes.data, 900)
            want = oracle.match_pair_port_test(imgs[0], imgs[1], ratio, mode)
            assert n == want.shape[0] and np.array_equal(out[:n], want), (mode, ratio)
    assert fn(imgs[0].ctypes.data, 900, imgs[1].ctypes.data, 1100, 0.6, 7, None, 0) < 0     # unknown test


def test_binary_key_cache_roundtrip_and_reference_reader(tmp_path):
    """<name>.bin in the layout of src/keys.cpp:551-648: written from a parsed text file, read back when the text file is gone,
    and byte for byte the file the UNMODIFIED in-bundler reader ReadKeyFileWithDesc was run on (stored with what it read)"""
    if not os.path.exists(KEYFILE):
        pytest.skip("shim/_build not built")
    lib = ctypes.CDLL(KEYFILE)
    rd = lib.bsfm_shim_read_key_file_info
    rd.restype = ctypes.c_int
    d = synth.sift_like_descriptors(1, [333], seed=9)[0]
    txt = str(tmp_path / "a.key")
    synth.write_key_file(txt, d, seed=3)
    kbuf, ibuf = ctypes.POINTER(ctypes.c_ubyte)(), ctypes.POINTER(ctypes.c_float)()
    n = rd(txt.encode(), ctypes.byref(kbuf), ctypes.byref(ibuf))
    assert n == 333
    keys = np.ctypeslib.as_array(kbuf, shape=(n * 128,)).reshape(n, 128).copy()
    info = np.ctypeslib.as_array(ibuf, shape=(n * 4,)).reshape(n, 4).copy()
    assert np.array_equal(keys, d)
    assert lib.bsfm_shim_write_key_bin((txt + ".bin").encode(), n, keys.ctypes.data_as(ctypes.c_void_p), info.ctypes.data_as(ctypes.c_void_p)) == 1
    os.remove(txt)                                   # only the cache is left: the reader falls through to <name>.bin
    kbuf2, ibuf2 = ctypes.POINTER(ctypes.c_ubyte)(), ctypes.POINTER(ctypes.c_float)()
    assert rd(txt.encode(), ctypes.byref(kbuf2), ctypes.byref(ibuf2)) == n
    assert np.array_equal(np.ctypeslib.as_array(kbuf2, shape=(n * 128,)).reshape(n, 128), d)
    assert np.array_equal(np.ctypeslib.as_array(ibuf2, shape=(n * 4,)).reshape(n, 4), info)
    g = np.load(REF_GOLD)                            # the reference's own reader on the file written by the same code
    assert hashlib.sha256(open(txt + ".bin", "rb").read()).hexdigest() == g["keybin_file_sha256"]
    assert g["keybin_ref_n"] == n
    assert g["keybin_ref_desc_sha256"] == _sha256(d) and np.array_equal(g["keybin_ref_xy"], info[:, :2])
