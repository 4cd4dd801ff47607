"""Loaders of committed golden fixtures shared by several test modules."""
import os
import types
from collections import namedtuple

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = os.path.join(GOLDEN, "movielens_multi_sparse.npz")
REFERENCE_ANSWERS = os.path.join(GOLDEN, "reference_answers.npz")

Feature = namedtuple("Feature", ["name", "index"])        # the reference's DataInfo column descriptor


def load_reference_answers():
    return np.load(REFERENCE_ANSWERS)


def load_feat_data_info():
    """The C1 DataInfo (DatasetFeat on sample_movielens_merged.csv, tests/golden/gen_movielens_feat.py)
    rebuilt from the golden files with the attributes the host and engine code read from it."""
    g = np.load(os.path.join(GOLDEN, "movielens_feat.npz"))
    a = load_reference_answers()
    n_users, n_items = int(g["n_users"]), int(g["n_items"])
    sparse_cols, dense_cols = a["di_sparse_col"].tolist(), a["di_dense_col"].tolist()

    def feature(cols, key):
        idx = [int(i) for i in g[key]]
        return Feature([cols[i] for i in idx], idx)

    id2item = {i: int(v) for i, v in enumerate(a["di_id2item"])}
    return types.SimpleNamespace(
        n_users=n_users, n_items=n_items,
        user_sparse_col=feature(sparse_cols, "user_sparse_col_index"),
        item_sparse_col=feature(sparse_cols, "item_sparse_col_index"),
        user_dense_col=feature(dense_cols, "user_dense_col_index"),
        item_dense_col=feature(dense_cols, "item_dense_col_index"),
        user_sparse_unique=g["user_sparse_unique"], item_sparse_unique=g["item_sparse_unique"],
        user_dense_unique=g["user_dense_unique"], item_dense_unique=None,
        col_name_mapping={"sparse_col": {c: i for i, c in enumerate(sparse_cols)},
                          "dense_col": {c: i for i, c in enumerate(dense_cols)}},
        sparse_idx_mapping={c: {v: i for i, v in enumerate(a[f"di_idx_mapping_{c}"].tolist())} for c in sparse_cols},
        sparse_offset=a["di_sparse_offset"], sparse_oov=a["di_sparse_oov"],
        id2item=id2item, item2id={v: k for k, v in id2item.items()},
        user_consumed={u: g["consumed_idx"][g["consumed_indptr"][u]:g["consumed_indptr"][u + 1]].tolist()
                       for u in range(n_users)})


def load_multi_sparse_spec():
    g = np.load(GOLD)
    spec = dict(
        n_users=int(g["n_users"]), n_items=int(g["n_items"]),
        user_sparse_col_index=g["user_sparse_col_index"].tolist(), item_sparse_col_index=g["item_sparse_col_index"].tolist(),
        user_dense_col_index=g["user_dense_col_index"].tolist(), item_dense_col_index=g["item_dense_col_index"].tolist(),
        user_sparse_unique=g["user_sparse_unique"], item_sparse_unique=g["item_sparse_unique"],
        user_dense_unique=g["user_dense_unique"].astype(np.float32), item_dense_unique=None,
        sparse_vocab=int(g["sparse_vocab"]),
        multi_sparse_combine_info=dict(field_offset=g["field_offset"].tolist(), field_len=g["field_len"].tolist(),
                                       feat_oov=g["feat_oov"]))
    spec["n_sparse"] = len(spec["user_sparse_col_index"]) + len(spec["item_sparse_col_index"])
    spec["n_dense"] = len(spec["user_dense_col_index"]) + len(spec["item_dense_col_index"])
    return g, spec
