"""Host logic of the recommendation shims: id re-mapping (construct_rec) and argument validation
(check_dynamic_rec_feats) and cold-start draws — compared with the answers of the unmodified reference
(libreco/recommendation/recommend.py:8-18,39-54, cold_start.py) stored in tests/golden/reference_answers.npz
(tests/golden/gen_reference_answers.py)."""
import types

import numpy as np
import pytest

from _fixtures import load_reference_answers

CONSTRUCT_USERS = [1, 2, 5, 4]
CHECK_ARGS = (("DeepFM", 1, None, [1]), ("DIN", [1, 2], {"a": 1}, None), ("DIN", 1, None, (1,)),
              ("DIN", 1, [1], None), ("YouTubeRanking", 1, None, [3, 4]))
COLD_USERS = ["u9", "u3", "u5"]
COLD_DEFAULT_RECS = np.arange(5, 25)


def _data_info(n_users=7, n_items=50, str_items=False):
    rng = np.random.default_rng(0)
    item_ids = rng.permutation(1000)[:n_items] + 5
    id2item = {i: (f"it{item_ids[i]}" if str_items else int(item_ids[i])) for i in range(n_items)}
    id2user = {u: 100 + 3 * u for u in range(n_users)}
    return types.SimpleNamespace(id2item=id2item, id2user=id2user)


@pytest.mark.parametrize("str_items", [False, True])
def test_construct_rec_maps_inner_to_original(str_items):
    from librecommender_b200.recommendation import construct_rec

    di = _data_info(str_items=str_items)
    rng = np.random.default_rng(1)
    users = [3, 0, 6]
    recs = rng.integers(0, 50, size=(3, 9))
    out = construct_rec(di, users, recs, inner_id=False)
    assert list(out) == [di.id2user[u] for u in users]
    for r, u in enumerate(users):
        want = [di.id2item[i] for i in recs[r]]
        assert out[di.id2user[u]].tolist() == want
    inner = construct_rec(di, users, recs, inner_id=True)
    for r, u in enumerate(users):
        np.testing.assert_array_equal(inner[u], recs[r])
    # second call reuses the cached lookup array and still follows a NEW mapping object
    di2 = _data_info(n_items=50, str_items=str_items)
    di2.id2item = {k: (v if str_items else v + 1) for k, v in di2.id2item.items()}
    out2 = construct_rec(di2, users, recs, inner_id=False)
    assert out2[di2.id2user[3]].tolist() == [di2.id2item[i] for i in recs[0]]


def construct_recs():
    return np.random.default_rng(2).integers(0, 50, size=(4, 12))


def test_construct_rec_equals_reference():
    from librecommender_b200.recommendation import construct_rec

    g = load_reference_answers()
    di = _data_info()
    for inner in (True, False):
        a = construct_rec(di, CONSTRUCT_USERS, construct_recs(), inner)
        assert list(a) == g[f"construct_{inner}_keys"].tolist()
        for k, want in zip(a, g[f"construct_{inner}_vals"]):
            np.testing.assert_array_equal(a[k], want)


def test_check_dynamic_rec_feats_errors():
    from librecommender_b200.recommendation import check_dynamic_rec_feats

    check_dynamic_rec_feats("DIN", 1, {"sex": "F"}, [1, 2, 3])          # fine
    with pytest.raises(ValueError, match="doesn't support arbitrary seq"):
        check_dynamic_rec_feats("DeepFM", 1, None, [1, 2])
    with pytest.raises(ValueError, match="Batch inference doesn't support assigning"):
        check_dynamic_rec_feats("DIN", [1, 2], {"sex": "F"}, None)
    with pytest.raises(ValueError, match="Batch inference doesn't support arbitrary item"):
        check_dynamic_rec_feats("DIN", [1, 2], None, [1, 2])
    with pytest.raises(ValueError, match="must be list or numpy"):
        check_dynamic_rec_feats("DIN", 1, None, (1, 2))
    with pytest.raises(ValueError, match="must be `dict`"):
        check_dynamic_rec_feats("DIN", 1, [("sex", "F")], None)
    # the reference's messages for the same arguments ("" where it accepts them)
    for args, ref_err in zip(CHECK_ARGS, load_reference_answers()["check_messages"].tolist(), strict=True):
        try:
            check_dynamic_rec_feats(*args)
            our_err = ""
        except ValueError as e:
            our_err = str(e)
        assert ref_err == our_err


def test_recommend_tf_feat_requires_engine_and_validates():
    from librecommender_b200 import _lib
    from librecommender_b200.recommendation import recommend_tf_feat

    model = types.SimpleNamespace(n_items=10, task="ranking", user_consumed={}, model_name="FM")
    with pytest.raises(_lib.B200Error):
        recommend_tf_feat(model, [0], 5, None, None, True, False)
    model.b200_engine = object()
    with pytest.raises(ValueError, match="Batch inference"):        # overrides are single-user only (recommend.py:39-54)
        recommend_tf_feat(model, [0, 1], 5, {"sex": "F"}, None, True, False)
    with pytest.raises(ValueError, match="exceeds num of items"):
        recommend_tf_feat(model, [0], 11, None, None, True, False)


def _cold_data_info(seed=7):
    rng_items = np.random.default_rng(3).permutation(500)[:40] + 1000
    di = types.SimpleNamespace(
        id2item={i: int(rng_items[i]) for i in range(40)}, item2id={int(rng_items[i]): i for i in range(40)},
        popular_items=[int(x) for x in rng_items[:15]], np_rng=np.random.default_rng(seed))
    return di


@pytest.mark.parametrize("strategy", ["average", "popular"])
@pytest.mark.parametrize("inner_id", [True, False])
def test_cold_start_rec_draws_like_the_reference(strategy, inner_id):
    """cold_start.py: one np_rng.choice(pool, n_rec) per user, in user order, with replacement."""
    from librecommender_b200.recommendation import cold_start_rec

    default_recs = COLD_DEFAULT_RECS
    users = COLD_USERS
    got = cold_start_rec(_cold_data_info(), default_recs, strategy, users, 6, inner_id)
    di = _cold_data_info()
    assert list(got) == users
    for u in users:
        if strategy == "average":
            picked = di.np_rng.choice(default_recs, 6)
            want = picked if inner_id else np.array([di.id2item[i] for i in picked])
        else:
            picked = di.np_rng.choice(di.popular_items, 6)
            want = np.array([di.item2id[i] for i in picked]) if inner_id else picked
        np.testing.assert_array_equal(got[u], want)
    for u, want in zip(users, load_reference_answers()[f"cold_{strategy}_{inner_id}"]):
        np.testing.assert_array_equal(got[u], want)
    with pytest.raises(ValueError, match="Unknown cold start strategy"):
        cold_start_rec(_cold_data_info(), default_recs, "nearest", users, 6, inner_id)
