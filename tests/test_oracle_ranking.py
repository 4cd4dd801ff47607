"""CPU: pin the oracle (numpy restatement) for the ranking path against
(a) the reference's own known-answer tests and (b) golden vectors produced by the
unmodified reference (tests/golden/gen_ranking.py)."""
import glob
import os

import numpy as np
import pytest

from oracle import ranking as orc
from _fixtures import load_reference_answers


def _dict_from_csr(indptr, idx):
    return {u: idx[indptr[u]:indptr[u + 1]].tolist()
            for u in range(len(indptr) - 1) if indptr[u + 1] > indptr[u]}


def test_known_answers_test_rank_reco():
    # vectors of reference tests/test_rank_reco.py:7-87
    user_ids = [1, 2]
    preds = np.array([-0.1, -0.01, 0, 0.1, 0.01, 1, -2, 4, 5, 6])
    consumed = {1: [3, 4], 2: [4]}
    with pytest.raises(ValueError):
        orc.rank_recommendations("ranking", user_ids, preds, 12, 5, consumed)
    ids = orc.rank_recommendations("ranking", user_ids, preds, 2, 5, consumed)
    np.testing.assert_array_equal(ids, [[2, 1], [3, 2]])
    ids = orc.rank_recommendations("ranking", user_ids, preds, 4, 5, consumed)  # cannot filter
    np.testing.assert_array_equal(ids, [[3, 4, 2, 1], [3, 2, 0, 1]])
    ids2d = orc.rank_recommendations("ranking", user_ids, preds.reshape(2, 5), 2, 5, consumed)
    np.testing.assert_array_equal(ids2d, [[2, 1], [3, 2]])
    _, scores = orc.rank_recommendations("ranking", user_ids, preds, 2, 5, consumed, True, True)
    assert (np.diff(scores, axis=1) <= 0).all()


def test_known_answers_consumed_dedup():
    # reference tests/test_consumed.py:12-25 and rust/src/utils.rs:46-57
    u = [1, 1, 1, 2, 2, 1, 2, 3, 2, 3]
    i = [11, 11, 999, 0, 11, 11, 999, 11, 999, 0]
    uc, ic = orc.build_consumed_unique(u, i)
    assert uc[1] == [11, 999, 11] and uc[2] == [0, 11, 999] and uc[3] == [11, 0]
    assert ic[11] == [1, 2, 1, 3] and ic[999] == [1, 2] and ic[0] == [2, 3]


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ranking_*.npz"))))
def test_rank_matches_reference_golden(path):
    g = np.load(path)
    consumed = _dict_from_csr(g["indptr"], g["idx"])
    uids = g["user_ids"].tolist()
    K, N = int(g["K"]), int(g["N"])
    np.testing.assert_array_equal(
        orc.rank_recommendations("ranking", uids, g["preds"], K, N, consumed, True), g["ids"])
    np.testing.assert_array_equal(
        orc.rank_recommendations("ranking", uids, g["preds"], K, N, consumed, False), g["ids_nofilter"])
    ids, sc = orc.rank_recommendations("ranking", uids, g["preds"].reshape(-1), K, N, consumed, True, True)
    np.testing.assert_array_equal(ids, g["ids_flat"])
    np.testing.assert_allclose(sc, g["scores_ranking"], rtol=1e-6)
    ids, sc = orc.rank_recommendations("rating", uids, g["preds"], K, N, consumed, True, True)
    np.testing.assert_array_equal(ids, g["ids_rating"])
    np.testing.assert_array_equal(sc, g["scores_rating"])


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "embed_*.npz"))))
def test_embed_matches_reference_golden(path):
    g = np.load(path)
    consumed = _dict_from_csr(g["indptr"], g["idx"])
    uids = g["user_ids"].tolist()
    K, N = int(g["K"]), int(g["N"])
    for flt, key in ((True, "ids"), (False, "ids_nofilter")):
        got = orc.recommend_from_embedding("ranking", uids, K, g["U"], g["I"], N, consumed, flt)
        ok = orc.near_tie_mask(g[key], got, g["full_scores"], rel_tol=1e-6)
        assert ok.all()
        assert (got == g[key]).mean() > 0.999


def random_rank_cases():
    rng = np.random.default_rng(5)
    for trial in range(20):
        B, N = int(rng.integers(1, 6)), int(rng.integers(5, 400))
        K = int(rng.integers(1, N + 1))
        preds = rng.standard_normal((B, N)).astype(np.float32)
        consumed = {u: rng.choice(N, size=int(rng.integers(0, N)), replace=False).tolist()
                    for u in range(B)}
        consumed = {u: v for u, v in consumed.items() if v}
        yield list(range(B)), preds, K, N, consumed


def test_oracle_vs_live_reference_random():
    """Random shapes and consumed lists against the reference's rank_recommendations
    (tests/golden/reference_answers.npz, tests/golden/gen_reference_answers.py)."""
    g = load_reference_answers()
    for trial, (uids, preds, K, N, consumed) in enumerate(random_rank_cases()):
        got = orc.rank_recommendations("ranking", uids, preds, K, N, consumed, True)
        np.testing.assert_array_equal(g[f"rank_{trial}"], got)


def test_assign_oov_and_predict():
    rng = np.random.default_rng(0)
    E = rng.standard_normal((5, 3)).astype(np.float32)
    out = orc.assign_embedding_oov(E)
    assert out.shape == (6, 3)
    np.testing.assert_allclose(out[-1], E.mean(axis=0))
    p = orc.predict_from_embedding(E, E, [0, 1], [2, 3])
    assert ((p > 0) & (p < 1)).all()


def test_numpy_path_variant_equals_deterministic_oracle():
    rng = np.random.default_rng(8)
    B, N, K = 6, 900, 25
    preds = rng.standard_normal((B, N)).astype(np.float32)
    consumed = {u: rng.choice(N, size=40, replace=False).tolist() for u in range(B - 1)}
    a = orc.rank_recommendations_numpy_path(list(range(B)), preds, K, N, consumed, True)
    b = orc.rank_recommendations("ranking", list(range(B)), preds, K, N, consumed, True)
    np.testing.assert_array_equal(a, b)
