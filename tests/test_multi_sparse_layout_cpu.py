"""Pins the multi-sparse LAYOUT assumptions against the reference's own pipeline
(tests/golden/movielens_multi_sparse.npz from examples/multi_sparse_example.py's columns):
* padding inside a multi-sparse field is the field's OOV index (feat_oov), fields follow the plain
  sparse columns (field_offset[0] == number of plain sparse columns);
* oracle.tf_models.row_features (user / item unique tables -> per-row index matrix) reproduces the
  reference's own TransformedSet.sparse_indices / dense_values for real training rows;
* `_spec_get` reads an object laid out like the reference's DataInfo;
* row_features equals the reference's prediction-time feed on both sample layouts (answers stored in
  tests/golden/reference_answers.npz by tests/golden/gen_reference_answers.py)."""
import types

import numpy as np
import pytest

from oracle import tf_models as tm

from _fixtures import Feature, load_feat_data_info, load_reference_answers  # noqa: E402
from _fixtures import load_multi_sparse_spec as load_spec  # noqa: E402


def test_layout_conventions():
    g, spec = load_spec()
    info = spec["multi_sparse_combine_info"]
    assert info["field_offset"] == [2] and info["field_len"] == [3]
    oov = int(info["feat_oov"][0])
    multi = spec["item_sparse_unique"]                      # all three item columns belong to the field
    assert (multi[-1] == oov).all()                         # OOV row
    assert (multi <= oov).all() and (multi == oov).any()    # padded sub-features use the OOV slot
    assert spec["user_sparse_col_index"] == [0, 1] and spec["item_sparse_col_index"] == [2, 3, 4]


def test_row_features_reproduce_reference_index_matrix():
    g, spec = load_spec()
    sparse, dense = tm.row_features(spec, g["train_users"], g["train_items"])
    np.testing.assert_array_equal(sparse, g["train_sparse"])
    np.testing.assert_allclose(dense, g["train_dense"], rtol=0, atol=0)


def test_spec_getter_reads_a_live_datainfo():
    """The multi-sparse sample layout as the reference's DataInfo holds it: column indices in
    ``Feature(name, index)`` descriptors (data_info.py:19-21,209-247), no item dense columns
    (``EmptyFeature``), the combine info as an attribute object."""
    from librecommender_b200.feat_models import _spec_get

    _, spec = load_spec()
    info = spec["multi_sparse_combine_info"]
    di = types.SimpleNamespace(
        n_users=spec["n_users"], n_items=spec["n_items"],
        user_sparse_col=Feature(["sex", "occupation"], spec["user_sparse_col_index"]),
        item_sparse_col=Feature(["genre1", "genre2", "genre3"], spec["item_sparse_col_index"]),
        user_dense_col=Feature(["age"], spec["user_dense_col_index"]), item_dense_col=Feature([], []),
        user_sparse_unique=spec["user_sparse_unique"], item_sparse_unique=spec["item_sparse_unique"],
        user_dense_unique=spec["user_dense_unique"], item_dense_unique=None,
        multi_sparse_combine_info=types.SimpleNamespace(**info))
    g = _spec_get(di)
    assert g("user_sparse_col_index") == list(di.user_sparse_col.index) == [0, 1]
    assert g("item_sparse_col_index") == list(di.item_sparse_col.index) == [2, 3, 4]
    assert g("user_dense_col_index") == list(di.user_dense_col.index) == [0]
    assert g("item_dense_col_index", []) in ([], None)
    assert g("n_users") == di.n_users and g("n_items") == di.n_items
    assert g("multi_sparse_combine_info").field_offset == [2]
    assert g("item_dense_unique") is None


@pytest.mark.parametrize("which", ["plain", "multi_sparse"])
def test_row_features_equal_reference_get_original_feats(which):
    """oracle.tf_models.row_features (the per-row feed the kernels reproduce from the unique tables)
    against the reference's own prediction-time function (prediction/preprocess.py:15-57) on the
    DataInfo of both sample layouts, incl. the OOV user / item rows."""
    from librecommender_b200.feat_models import _spec_get

    g = _spec_get(load_spec()[1] if which == "multi_sparse" else load_feat_data_info())
    spec = {k: g(k) for k in ("n_users", "n_items", "user_sparse_unique", "item_sparse_unique", "user_dense_unique",
                              "item_dense_unique")}
    for k in ("user_sparse_col_index", "item_sparse_col_index", "user_dense_col_index", "item_dense_col_index"):
        spec[k] = g(k) or []
    spec["n_sparse"] = len(spec["user_sparse_col_index"]) + len(spec["item_sparse_col_index"])
    spec["n_dense"] = len(spec["user_dense_col_index"]) + len(spec["item_dense_col_index"])
    ref = load_reference_answers()
    users, items = ref[f"rowfeat_{which}_users"], ref[f"rowfeat_{which}_items"]
    assert users[-1] == spec["n_users"] and items[-1] == spec["n_items"]
    sparse, dense = tm.row_features(spec, users, items)
    np.testing.assert_array_equal(sparse, ref[f"rowfeat_{which}_sparse"])
    np.testing.assert_array_equal(dense, ref[f"rowfeat_{which}_dense"])
