"""CPU tests (no GPU): pin the MATCH oracle restatement (oracle/match_oracle.c) against the golden
vectors produced by the unmodified reference (tests/golden/make_match_golden.py) and against its stored results on further
inputs (tests/golden/make_reference_golden.py)."""
import os

import numpy as np
import pytest

from bundler_sfm_b200 import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden", "match_golden.npz")
REF_GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def ref_gold():
    return np.load(REF_GOLD)


def test_port_matches_golden_sift_pairs(oracle, gold):
    for i in range(4):
        for j in range(i):
            got = oracle.match_pair_port(gold[f"sift_img{j}"], gold[f"sift_img{i}"], 0.6)
            assert np.array_equal(got, gold[f"sift_exact_{j}_{i}"]), (j, i)


def test_port_matches_golden_edge_cases(oracle, gold):
    names = sorted({k[len("edge_"):-2] for k in gold.files if k.startswith("edge_") and k.endswith("_q")})
    assert len(names) >= 10
    for name in names:
        q, db = gold[f"edge_{name}_q"], gold[f"edge_{name}_db"]
        for tag, ratio in (("m06", 0.6), ("m09", 0.9)):
            got = oracle.match_pair_port(q, db, ratio)
            assert np.array_equal(got, gold[f"edge_{name}_{tag}"]), (name, tag)


def test_golden_edge_semantics(gold):
    # single database key: d1 = INT_MAX so (almost) every query matches index 0 (SURVEY.md H6)
    m = gold["edge_n2_is_1_m06"]
    assert m.shape[0] == 7 and np.all(m[:, 1] == 0)
    # tie for best never matches
    assert gold["edge_tie_best_m06"].shape[0] == 0
    # identical descriptors: d0 = 0 < 0.36*d1 whenever d1 > 0
    assert gold["edge_identical_m06"].shape[0] == 10
    # ratio boundary, integer form 25*d0 < 9*d1: (9,25)->no, (9,26)->yes, (10,25)->no, (36,100)->no, (35,100)->yes, (36,101)->yes
    expect = [0, 1, 0, 0, 1, 1]
    for k, e in enumerate(expect):
        assert gold[f"edge_ratio_boundary_{k}_m06"].shape[0] == e, k


def test_cap200_recall_informational(gold):
    # the stock 200-visit cap is approximate; report recall of exact matches (not a gate)
    tot = hit = 0
    for i in range(4):
        for j in range(i):
            ex = {tuple(r) for r in gold[f"sift_exact_{j}_{i}"]}
            ap = {tuple(r) for r in gold[f"sift_cap200_{j}_{i}"]}
            tot += len(ex); hit += len(ex & ap)
    assert tot > 0 and hit / tot > 0.5


def test_port_vs_reference_random(oracle, ref_gold):
    for seed in range(3):
        imgs = synth.sift_like_descriptors(2, [300 + 17 * seed, 280], seed=100 + seed)
        a = oracle.match_pair_port(imgs[0], imgs[1], 0.6)
        assert np.array_equal(a, ref_gold[f"matchrnd{seed}_sift"])
        u1, u2 = synth.random_descriptors(90, seed), synth.random_descriptors(75, seed + 50)
        assert np.array_equal(oracle.match_pair_port(u1, u2, 0.95), ref_gold[f"matchrnd{seed}_uniform"])


def test_all_pairs_table_format(oracle):
    imgs = synth.sift_like_descriptors(4, [200, 0, 180, 190], seed=3)
    txt, counts = oracle.match_all_pairs_port(imgs, -1, 0.6, 16)
    lines = txt.split("\n")
    assert lines[-1] == ""
    # header "j i", count, then count lines; only pairs with >= 16 matches, j < i, empty image skipped
    pos = 0
    seen = []
    while pos < len(lines) - 1:
        j, i = map(int, lines[pos].split())
        c = int(lines[pos + 1])
        assert c >= 16 and j < i and j != 1 and i != 1
        assert counts[i, j] == c
        seen.append((j, i))
        pos += 2 + c
    assert seen == sorted(seen, key=lambda p: (p[1], p[0]))
    # windowed variant only visits j >= i - window
    txt_w, counts_w = oracle.match_all_pairs_port(imgs, 1, 0.6, 16)
    assert counts_w[3, 0] == 0 and counts_w[3, 2] == counts[3, 2]


def test_port_keys_cpp_test_mode_vs_reference_exhaustive(ref_gold):
    """oracle/match_oracle.c mode 1 (sqrt(d0/d1) <= ratio, `registered` subset) against the stored results of the UNMODIFIED
    MatchKeysExhaustive of src/keys.cpp: the pair of calls bundler --add_images makes (Bundle.cpp:3812-3820)"""
    from oracle import loader
    imgs = synth.sift_like_descriptors(2, [600, 750], seed=11)
    extra = np.where(np.random.default_rng(3).random(750) < 0.6, 5, -1).astype(np.int32)
    for q, (reg, ratio) in enumerate(((True, 0.75), (False, 1.0), (False, 0.6), (True, 0.9))):
        want = ref_gold[f"keyscpp{q}_matches"]
        got = loader.match_pair_port_test(imgs[0], imgs[1], ratio, 1, extra, reg)
        assert np.array_equal(got, want), (reg, ratio)
        assert want.shape[0] > 0
    # (a database of ONE key is a fatal error in the reference: ANN aborts with "Requesting more near neighbors than data
    #  points", lib/ann_1.1_char/src/kd_search.cpp -- not a case to compare)


def test_port_on_real_sift_descriptors_kermit_golden():
    """real SIFT descriptors of the reference's example set (examples/kermit, 11 images, 55 pairs): the C restatement against
    the stored exact-mode output of the unmodified reference (tests/golden/kermit_match_golden.npz)"""
    from oracle import loader
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "kermit_match_golden.npz"))
    n = int(g["num_images"])
    descs = [g[f"desc{i}"] for i in range(n)]
    pos, q = 0, 0
    for i in range(n):
        for j in range(i):
            c = int(g["counts"][q])
            assert np.array_equal(loader.match_pair_port(descs[j], descs[i], 0.6), g["matches"][pos:pos + c]), (j, i)
            pos += c; q += 1
    for (a, b) in ((0, 1), (3, 7), (10, 9)):
        assert np.array_equal(loader.match_pair_port_test(descs[a], descs[b], 0.75, 1), g[f"keys_{a}_{b}"])
