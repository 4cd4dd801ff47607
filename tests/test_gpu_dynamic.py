"""GPU: the a3 / a15 gaps closed in round 2, on the reference's own C1 data pipeline (DatasetFeat on
sample_movielens_merged.csv, examples/feat_ranking_example.py:27-41; its DataInfo and the reference's
feeds are stored in tests/golden/movielens_feat.npz and tests/golden/reference_answers.npz):

* single-user ``recommend_tf_feat`` with ``user_feats`` / ``seq`` supplied for the call
  (recommendation/recommend.py:39-54,81-105) == the numpy restatement of the model graph evaluated on
  the reference's own tiled + overridden feed (``_get_original_feats`` + ``set_temp_feats``);
* ``assign_oov`` on the device tables == the restated ``assign_tf_variables_oov`` rule, and
  ``default_recs`` == top-2000 of the OOV user without the consumed filter (bases/tf_base.py:145-153).
The TF graph math itself stays parity-unpinned (no TensorFlow anywhere); the FEED is the reference's."""
import types

import numpy as np
import pytest

from _fixtures import load_feat_data_info, load_reference_answers

pytestmark = pytest.mark.gpu


def override_cases(n_users):
    return ((5, {"sex": "F", "age": 40.0}), (11, {"occupation": 3}), (n_users, {"age": 18.0}))


@pytest.fixture(scope="module")
def di():
    return load_feat_data_info()


def _spec(di):
    spec = dict(n_users=di.n_users, n_items=di.n_items,
                user_sparse_col_index=list(di.user_sparse_col.index), item_sparse_col_index=list(di.item_sparse_col.index),
                user_dense_col_index=list(di.user_dense_col.index), item_dense_col_index=list(di.item_dense_col.index),
                user_sparse_unique=di.user_sparse_unique, item_sparse_unique=di.item_sparse_unique,
                user_dense_unique=di.user_dense_unique.astype(np.float32), item_dense_unique=None,
                sparse_vocab=int(max(di.user_sparse_unique.max(), di.item_sparse_unique.max()) + 1))
    spec["n_sparse"] = len(spec["user_sparse_col_index"]) + len(spec["item_sparse_col_index"])
    spec["n_dense"] = len(spec["user_dense_col_index"]) + len(spec["item_dense_col_index"])
    return spec


@pytest.mark.parametrize("name", ["FM", "DeepFM"])
def test_single_user_feature_override_matches_reference_feed(di, name):
    from librecommender_b200 import feat_models as fm
    from librecommender_b200.recommendation import recommend_tf_feat
    from oracle import ranking as orc
    from oracle import tf_models as tm

    spec = _spec(di)
    rng = np.random.default_rng(3)
    if name == "FM":
        w, fwd = tm.make_fm_weights(rng, spec, 16, use_bn=True), tm.fm_forward
    else:
        w, fwd = tm.make_deepfm_weights(rng, spec, 16, (64, 32), True), tm.deepfm_forward
    engine = getattr(fm, name)(spec, w, di.user_consumed)
    model = types.SimpleNamespace(b200_engine=engine, n_items=di.n_items, n_users=di.n_users, task="ranking",
                                  data_info=di, user_consumed=di.user_consumed, model_name=name)
    N = di.n_items
    ref_feed = load_reference_answers()
    for c, (user, feats) in enumerate(override_cases(di.n_users)):
        sp, de = ref_feed["feed_sparse"][c], ref_feed["feed_dense"][c]           # the reference's own feed
        preds = fwd(w, np.repeat(user, N), np.arange(N), sp.astype(np.int64), de.astype(np.float32),
                    dtype=np.float64).astype(np.float32)
        for n_rec in (7, 50):
            got = recommend_tf_feat(model, [user], n_rec, feats, None, True, False, inner_id=True)
            ref = orc.rank_recommendations("ranking", [user], preds, n_rec, N, di.user_consumed, True)
            assert got.shape == (1, n_rec)
            assert orc.near_tie_mask(ref, got, preds.reshape(1, N), 1e-5).all()
        # the override really changes the scores (otherwise the test proves nothing)
        base = engine.score_all_items(__import__("torch").tensor([user], device=engine.device)).cpu().numpy()[0]
        assert np.abs(base - preds).max() > 1e-4
    with pytest.raises(ValueError):
        recommend_tf_feat(model, [1, 2], 5, {"age": 3.0}, None, True, False, inner_id=True)


def test_assign_oov_and_default_recs(di):
    from librecommender_b200 import feat_models as fm
    from librecommender_b200.dynamic_feats import assign_oov_rows
    from oracle import ranking as orc
    from oracle import tf_models as tm

    spec = _spec(di)
    w = tm.make_fm_weights(np.random.default_rng(9), spec, 16, use_bn=True)
    engine = fm.FM(spec, w, di.user_consumed)
    engine.assign_oov(di.sparse_oov)
    w2 = assign_oov_rows(w, di.n_users, di.n_items, di.sparse_oov)
    for k in ("user_embeds", "item_embeds", "sparse_embeds", "user_linear", "item_linear", "sparse_linear"):
        np.testing.assert_allclose(engine.t[k].cpu().numpy().reshape(np.asarray(w2[k]).shape), w2[k], rtol=2e-6, atol=1e-7)
    N = di.n_items
    n_rec = min(2000, N)
    got = engine.default_recs()
    uu, ii = np.repeat(di.n_users, N), np.arange(N)
    sp, de = tm.row_features(spec, uu, ii)
    preds = tm.fm_forward(w2, uu, ii, sp, de, dtype=np.float64).astype(np.float32)
    ref = orc.rank_recommendations("ranking", [di.n_users], preds, n_rec, N, di.user_consumed, False)
    assert got.shape == (n_rec,)
    assert orc.near_tie_mask(ref, got[None, :], preds.reshape(1, N), 1e-5).all()
