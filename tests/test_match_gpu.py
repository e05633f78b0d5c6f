"""GPU parity tests of the MATCH path: every call goes through the C ABI (libbsfm_b200.so) and is
compared bit-exactly with the CPU oracle (oracle/match_oracle.c, pinned to the reference by
tests/test_oracle_match.py) and with the committed golden vectors of the unmodified reference."""
import os

import numpy as np
import pytest

from bundler_sfm_b200 import keymatch, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "match_golden.npz")
# every kernel variant of the library runs the whole suite:
#   tc       tcgen05 kernel, bound epilogue, one CTA per unit, two accumulator stages of 256 columns
#   tc_quad  the same with four accumulator stages of 128 columns
#   tc_exact tcgen05 kernel, exact chunk-minimum epilogue (also the path of images > 8192 rows)
#   tc_pair  tcgen05 cta_group::2 kernel on CTA pairs
#   dp4a     CUDA-core kernel
KERNELS = {"tc": {"BSFM_MATCH_KERNEL": "0", "BSFM_MATCH_QUAD": "0"},
           "tc_quad": {"BSFM_MATCH_KERNEL": "0", "BSFM_MATCH_QUAD": "1"},
           "tc_exact": {"BSFM_MATCH_KERNEL": "0", "BSFM_MATCH_EPILOGUE": "0"},
           "tc_pair": {"BSFM_MATCH_KERNEL": "0", "BSFM_MATCH_PAIR": "1"},
           "dp4a": {"BSFM_MATCH_KERNEL": "1"}}


@pytest.fixture(params=list(KERNELS))
def kernel(request, monkeypatch):
    for k in ("BSFM_MATCH_KERNEL", "BSFM_MATCH_EPILOGUE", "BSFM_MATCH_PAIR", "BSFM_MATCH_QUAD"):
        monkeypatch.delenv(k, raising=False)
    for k, v in KERNELS[request.param].items():
        monkeypatch.setenv(k, v)
    return request.param


def test_golden_sift_pairs(kernel):
    gold = np.load(GOLD)
    for i in range(4):
        for j in range(i):
            got = keymatch.match_keys(gold[f"sift_img{j}"], gold[f"sift_img{i}"], 0.6)
            assert np.array_equal(got, gold[f"sift_exact_{j}_{i}"]), (kernel, j, i)


def test_golden_edge_cases(kernel):
    gold = np.load(GOLD)
    names = sorted({k[len("edge_"):-2] for k in gold.files if k.startswith("edge_") and k.endswith("_q")})
    for name in names:
        q, db = gold[f"edge_{name}_q"], gold[f"edge_{name}_db"]
        for tag, ratio in (("m06", 0.6), ("m09", 0.9)):
            got = keymatch.match_keys(q, db, ratio)
            assert np.array_equal(got, gold[f"edge_{name}_{tag}"]), (kernel, name, tag)


@pytest.mark.parametrize("n1,n2", [(1, 1), (1, 2), (5, 3), (128, 256), (129, 257), (1000, 777), (2500, 5000), (300, 9000)])
def test_pair_vs_oracle_sizes(kernel, oracle, n1, n2):
    imgs = synth.sift_like_descriptors(2, [n1, n2], seed=n1 * 7 + n2)
    got = keymatch.match_keys(imgs[0], imgs[1], 0.6)
    want = oracle.match_pair_port(imgs[0], imgs[1], 0.6)
    assert np.array_equal(got, want)


def test_uniform_random_and_loose_ratio(kernel, oracle):
    a, b = synth.random_descriptors(700, 1), synth.random_descriptors(900, 2)
    for ratio in (0.6, 0.95, 0.999):
        assert np.array_equal(keymatch.match_keys(a, b, ratio), oracle.match_pair_port(a, b, ratio)), ratio


def test_empty_inputs(kernel):
    z = np.zeros((0, 128), np.uint8)
    k = synth.random_descriptors(10, 3)
    assert keymatch.match_keys(z, k).shape == (0, 2)
    assert keymatch.match_keys(k, z).shape == (0, 2)


def test_all_pairs_table_identical_to_oracle(kernel, oracle):
    # ragged sizes incl. an empty image and images smaller than a tile; KeyMatchFull order + >=16 filter
    sizes = [600, 0, 300, 17, 513, 256, 1, 700]
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=21)
    for window in (-1, 2):
        pairs, counts, matches = keymatch.key_match_full(imgs, window, 0.6)
        txt = keymatch.format_match_table(pairs, counts, matches, 16)
        want_txt, want_counts = oracle.match_all_pairs_port(imgs, window, 0.6, 16)
        for (j, i), c in zip(pairs, counts):
            assert want_counts[i, j] == c, (window, j, i)
        assert txt == want_txt
        assert counts.sum() == matches.shape[0]


def test_sharded_runs_concatenate(kernel, oracle):
    sizes = [400, 380, 390, 410, 300, 420]
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=5)
    keys, key_off = keymatch.concat_keys(imgs)
    db = keymatch.KeyDatabase(keys, key_off)
    db.run(0, len(sizes), -1, 0.6)
    c_all, m_all = db.fetch()
    parts_c, parts_m = [], []
    for b, e in keymatch.shard_images(sizes, -1, 3):
        db.run(b, e, -1, 0.6)
        c, m = db.fetch()
        parts_c.append(c); parts_m.append(m)
    db.close()
    assert np.array_equal(np.concatenate(parts_c), c_all)
    assert np.array_equal(np.concatenate(parts_m), m_all)


def test_chunked_launches_equal_single_launch(kernel, monkeypatch):
    sizes = [900, 800, 1000, 700]
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=9)
    ref = keymatch.key_match_full(imgs, -1, 0.6)
    monkeypatch.setenv("BSFM_MATCH_CHUNK_MSLOTS", "1")   # 1 Mi slots/launch; forces several launches? (small here)
    got = keymatch.key_match_full(imgs, -1, 0.6)
    assert np.array_equal(ref[1], got[1]) and np.array_equal(ref[2], got[2])


def test_tc_equals_dp4a_at_scale(monkeypatch):
    """size-independent property at a scale the CPU oracle cannot check in seconds: the tensor-core
    kernel and the independent DP4A kernel must produce the identical match stream, and the table
    must satisfy the invariants of the algorithm (ascending query index inside a pair, in-range ids)."""
    sizes = [5000] * 12
    imgs = synth.sift_like_descriptors(len(sizes), sizes, seed=7)
    for k in ("BSFM_MATCH_KERNEL", "BSFM_MATCH_EPILOGUE", "BSFM_MATCH_PAIR"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("BSFM_MATCH_KERNEL", "0")
    p0, c0, m0 = keymatch.key_match_full(imgs, -1, 0.6)
    monkeypatch.setenv("BSFM_MATCH_KERNEL", "1")
    p1, c1, m1 = keymatch.key_match_full(imgs, -1, 0.6)
    assert np.array_equal(c0, c1) and np.array_equal(m0, m1)
    # the other two tensor-core variants at the same scale
    monkeypatch.setenv("BSFM_MATCH_KERNEL", "0")
    for extra in ({"BSFM_MATCH_EPILOGUE": "0"}, {"BSFM_MATCH_PAIR": "1"}):
        for k, v in extra.items():
            monkeypatch.setenv(k, v)
        p2, c2, m2 = keymatch.key_match_full(imgs, -1, 0.6)
        assert np.array_equal(c0, c2) and np.array_equal(m0, m2), extra
        for k in extra:
            monkeypatch.delenv(k)
    assert m0.shape[0] > 1000
    pos = 0
    for (j, i), c in zip(p0, c0):
        blk = m0[pos:pos + c]
        assert np.all(np.diff(blk[:, 0]) > 0)
        assert blk[:, 0].min(initial=0) >= 0 and blk[:, 0].max(initial=0) < sizes[j]
        assert blk[:, 1].min(initial=0) >= 0 and blk[:, 1].max(initial=0) < sizes[i]
        pos += c
    # consecutive images share 30% noisy copies -> those pairs must be rich in matches
    for (j, i), c in zip(p0, c0):
        if i == j + 1:
            assert c > 500


def test_config4_table_sampled_pairs_vs_oracle_and_reference_exact(oracle):
    """BASELINE.json configs[3] at full size (500 images x 5000 keys, 124,750 pairs): 200 randomly drawn image pairs of the
    GPU table are compared with the CPU oracle (pinned to the reference), and a handful of them with the stored output of the
    UNMODIFIED reference MatchKeys in exact mode (max_pts_visit = 0, keys2a.cpp:347-372; tests/golden/reference_golden.npz)."""
    N, K = 500, 5000
    imgs = synth.sift_like_descriptors(N, K, seed=7)
    pairs, counts, matches = keymatch.key_match_full(imgs, -1, 0.6)
    assert len(pairs) == N * (N - 1) // 2 and int(counts.sum()) == matches.shape[0] == 1068340
    starts = np.concatenate([[0], np.cumsum(counts)])
    rng = np.random.default_rng(2026)
    picked = rng.choice(len(pairs), 200, replace=False)
    # make sure rich pairs (consecutive images share 30 % noisy copies) are represented, not only sparse ones
    rich = [q for q, (j, i) in enumerate(pairs) if i == j + 1][::25]
    picked = np.unique(np.concatenate([picked, np.array(rich[:20], dtype=picked.dtype)]))
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz"))
    ref_pairs = [tuple(int(v) for v in p) for p in g["config4_pairs"]]
    ref_starts = np.concatenate([[0], np.cumsum(g["config4_counts"])])
    nref = 0
    for q in picked:
        j, i = pairs[q]
        got = matches[starts[q]:starts[q + 1]]
        want = oracle.match_pair_port(imgs[j], imgs[i], 0.6)
        assert np.array_equal(got, want), (j, i)
        if nref < 3 or (i == j + 1 and nref < 6):
            assert ref_pairs[nref] == (j, i)
            assert np.array_equal(got, g["config4_matches"][ref_starts[nref]:ref_starts[nref + 1]]), ("reference exact mode", j, i)
            nref += 1
    assert nref == len(ref_pairs) >= 3


def test_kermit_real_sift_table_equals_reference(kernel):
    """BASELINE.json configs[0]'s MATCH stage on REAL descriptors: OpenCV-SIFT keys of the 11 kermit images, all 55 pairs, against
    the stored exact-mode table of the unmodified reference (tests/golden/kermit_match_golden.npz, made by
    make_kermit_match_golden.py); real data has near-duplicate keys and clipped descriptors that the synthetic sets lack"""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "kermit_match_golden.npz"))
    descs = [g[f"desc{i}"] for i in range(int(g["num_images"]))]
    pairs, counts, matches = keymatch.key_match_full(descs, -1, 0.6)
    assert np.array_equal(counts, g["counts"]) and np.array_equal(matches, g["matches"])
    assert (counts >= 16).sum() == 30
