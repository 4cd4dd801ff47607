"""Host-side inference plumbing against the UNMODIFIED reference, whose answers on the C1 DataInfo
(DatasetFeat on sample_movielens_merged.csv) are stored in tests/golden/reference_answers.npz
(tests/golden/gen_reference_answers.py): per-row features of "one user x every item" with user features
overridden (recommendation/preprocess.py:104-212 + prediction/preprocess.py:58-104), the padded sequence
row (recommendation/preprocess.py:36-45) and the OOV-row assignment rule (bases/tf_base.py:310-353,
restated because it is a TensorFlow graph op)."""
import numpy as np
import pytest

from _fixtures import load_feat_data_info, load_reference_answers

FEATS = [None, {"sex": "F", "age": 33.0}, {"occupation": 17, "nonexistent": 1},
         {"sex": "no-such-value", "age": 5.0, "genre1": "Comedy"}]


def users(n_users):
    return (0, 7, n_users)                                      # incl. the OOV user row


def rec_seq_cases(id2item):
    some = [id2item[i] for i in range(25)]
    return ((list(range(3)), True), (list(range(40)), True), (some, False), (some[:4] + ["unknown"], False))


@pytest.fixture(scope="module")
def data_info():
    return load_feat_data_info()


@pytest.fixture(scope="module")
def golden():
    return load_reference_answers()


@pytest.mark.parametrize("feats", FEATS)
def test_dynamic_feature_rows_equal_reference(data_info, golden, feats):
    from librecommender_b200.dynamic_feats import dynamic_feature_rows

    f = FEATS.index(feats)
    assert golden["dyn_feats"][f] == repr(feats)
    rows = golden["dyn_rows"]                                   # a fixed sample of the N item rows
    for j, user in enumerate(users(data_info.n_users)):
        case = f * 3 + j
        before = (data_info.user_sparse_unique.copy(), data_info.user_dense_unique.copy())
        sp, de = dynamic_feature_rows(data_info, user, feats)
        assert sp.shape[0] == de.shape[0] == data_info.n_items
        np.testing.assert_array_equal(sp[rows], golden["dyn_sparse"][case])
        np.testing.assert_array_equal(de[rows], golden["dyn_dense"][case])
        np.testing.assert_array_equal(data_info.user_sparse_unique, before[0])      # nothing was modified
        np.testing.assert_array_equal(data_info.user_dense_unique, before[1])


def test_build_rec_seq_equals_reference(data_info, golden):
    from librecommender_b200.dynamic_feats import build_rec_seq

    for c, (seq, inner) in enumerate(rec_seq_cases(data_info.id2item)):
        ref_seq, ref_len = golden["rec_seq"][c], golden["rec_seq_len"][c]
        got_seq, got_len = build_rec_seq(seq, data_info.n_items, 10, data_info.item2id, inner)
        np.testing.assert_array_equal(got_seq, ref_seq)
        np.testing.assert_array_equal(got_len, ref_len)
        assert [str(got_seq.dtype), str(got_len.dtype)] == golden["rec_seq_dtypes"].tolist()


def test_assign_oov_rows_rule(data_info):
    from librecommender_b200.dynamic_feats import assign_oov_rows

    rng = np.random.default_rng(0)
    nu, ni = data_info.n_users, data_info.n_items
    oov = data_info.sparse_oov
    V = int(max(oov)) + 1
    w = dict(user_embeds=rng.standard_normal((nu + 1, 4)).astype(np.float32),
             item_embeds=rng.standard_normal((ni + 1, 4)).astype(np.float32),
             user_linear=rng.standard_normal(nu + 1).astype(np.float32),
             sparse_embeds=rng.standard_normal((V, 4)).astype(np.float32),
             sparse_linear=rng.standard_normal(V).astype(np.float32))
    out = assign_oov_rows(w, nu, ni, oov)
    np.testing.assert_allclose(out["user_embeds"][nu], w["user_embeds"][:nu].mean(0), rtol=1e-6)
    np.testing.assert_allclose(out["item_embeds"][ni], w["item_embeds"][:ni].mean(0), rtol=1e-6)
    np.testing.assert_allclose(out["user_linear"][nu], w["user_linear"][:nu].mean(), rtol=1e-6)
    start = 0
    for o in oov:                                             # tf_base.py:336-349
        if start >= o:
            continue
        np.testing.assert_allclose(out["sparse_embeds"][o], w["sparse_embeds"][start:o].mean(0), rtol=1e-6)
        np.testing.assert_allclose(out["sparse_linear"][o], w["sparse_linear"][start:o].mean(), rtol=1e-6)
        start = o + 1
    keep = np.setdiff1d(np.arange(V), np.asarray(oov))
    np.testing.assert_array_equal(out["sparse_embeds"][keep], w["sparse_embeds"][keep])   # only oov rows change
    np.testing.assert_array_equal(w["user_embeds"][nu], w["user_embeds"][nu])             # input dict untouched
