"""Answers of the UNMODIFIED reference for the tests that compare with it directly (host recommendation
shims, dynamic feature rows, the per-row feed of both sample layouts, ranking and sampling streams, the
on-disk default_recs format), plus the pieces of the C1 DataInfo (DatasetFeat on
sample_movielens_merged.csv, examples/feat_ranking_example.py:27-41) those tests read beyond
tests/golden/movielens_feat.npz.  Inputs come from the test modules themselves, so a test and its
golden answer cannot drift apart.

    python tests/golden/gen_reference_answers.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path.insert(0, ROOT)
sys.path.insert(0, TESTS)
from oracle.ref_loader import REFERENCE_ROOT, load_reference  # noqa: E402

load_reference()
from libreco.data import DatasetFeat, split_by_ratio_chrono  # noqa: E402
from libreco.prediction.preprocess import get_original_feats, set_temp_feats  # noqa: E402
from libreco.recommendation import rank_recommendations  # noqa: E402
from libreco.recommendation.cold_start import cold_start_rec  # noqa: E402
from libreco.recommendation.preprocess import _get_original_feats, build_rec_seq  # noqa: E402
from libreco.recommendation.recommend import check_dynamic_rec_feats, construct_rec  # noqa: E402
from libreco.sampling.negatives import negatives_from_random  # noqa: E402
from libreco.utils.save_load import save_default_recs  # noqa: E402

import test_construct_rec_cpu as t_rec  # noqa: E402
import test_dynamic_feats_cpu as t_dyn  # noqa: E402
import test_gpu_dynamic as t_gdyn  # noqa: E402
import test_oracle_ranking as t_rank  # noqa: E402
import test_sampling_cpu as t_smp  # noqa: E402


def feat_data_info():
    data = pd.read_csv(os.path.join(REFERENCE_ROOT, "examples/sample_data/sample_movielens_merged.csv"))
    train, _ = split_by_ratio_chrono(data, test_size=0.2)
    _, di = DatasetFeat.build_trainset(train, ["sex", "age", "occupation"], ["genre1", "genre2", "genre3"],
                                       ["sex", "occupation", "genre1", "genre2", "genre3"], ["age"])
    return di


def multi_sparse_data_info():
    spec_ = importlib.util.spec_from_file_location("gen_ms", os.path.join(HERE, "gen_movielens_multi_sparse.py"))
    mod = importlib.util.module_from_spec(spec_)
    sys.modules["gen_ms"] = mod
    spec_.loader.exec_module(mod)
    return mod.build()[1]


def data_info_pieces(di, out):
    """What dynamic_feature_rows / build_rec_seq / assign_oov read from a DataInfo, beyond movielens_feat.npz."""
    cm = di.col_name_mapping
    for kind in ("sparse_col", "dense_col"):
        assert list(cm[kind].values()) == list(range(len(cm[kind])))
        out[f"di_{kind}"] = np.array(list(cm[kind]))
    for col, mapping in di.sparse_idx_mapping.items():
        assert list(mapping.values()) == list(range(len(mapping)))
        out[f"di_idx_mapping_{col}"] = np.array(list(mapping))
    out["di_sparse_offset"] = np.asarray(di.sparse_offset)
    out["di_sparse_oov"] = np.asarray(di.sparse_oov)
    out["di_id2item"] = np.array([di.id2item[i] for i in range(di.n_items)])


def dynamic_rows(di, out):
    rows = np.sort(np.random.default_rng(0).choice(di.n_items, 64, replace=False))
    out["dyn_rows"] = np.append(rows, di.n_items - 1)
    out["dyn_feats"] = np.array([repr(f) for f in t_dyn.FEATS])
    sps, des = [], []
    for feats in t_dyn.FEATS:
        for user in t_dyn.users(di.n_users):
            sp, de = _get_original_feats(di, user, di.n_items, True, True)
            if feats is not None:
                sp, de = set_temp_feats(di, sp, de, feats)
            sps.append(sp[out["dyn_rows"]])
            des.append(de[out["dyn_rows"]])
    out["dyn_sparse"], out["dyn_dense"] = np.stack(sps), np.stack(des)
    model = types.SimpleNamespace(data_info=di, n_items=di.n_items, max_seq_len=10)
    seqs, lens = [], []
    for seq, inner in t_dyn.rec_seq_cases(di.id2item):
        s, n = build_rec_seq(seq, model, inner)
        seqs.append(s)
        lens.append(n)
    out["rec_seq"], out["rec_seq_len"] = np.stack(seqs), np.stack(lens)
    out["rec_seq_dtypes"] = np.array([str(seqs[0].dtype), str(lens[0].dtype)])
    # full feeds of the GPU override cases (one user x every item)
    sps, des = [], []
    for user, feats in t_gdyn.override_cases(di.n_users):
        sp, de = _get_original_feats(di, user, di.n_items, True, True)
        sp, de = set_temp_feats(di, sp, de, feats)
        sps.append(sp.astype(np.int32))
        des.append(de.astype(np.float32))
    out["feed_sparse"], out["feed_dense"] = np.stack(sps), np.stack(des)


def row_features(which, di, out):
    rng = np.random.default_rng(0)
    users = np.concatenate([rng.integers(0, di.n_users, 500), [di.n_users]])      # + the OOV user row
    items = np.concatenate([rng.integers(0, di.n_items, 500), [di.n_items]])
    _, _, sparse, dense = get_original_feats(di, users, items, True, True)
    out[f"rowfeat_{which}_users"], out[f"rowfeat_{which}_items"] = users, items
    out[f"rowfeat_{which}_sparse"], out[f"rowfeat_{which}_dense"] = sparse, dense


def recommendation_shims(out):
    di = t_rec._data_info()
    for inner in (True, False):
        rec = construct_rec(di, t_rec.CONSTRUCT_USERS, t_rec.construct_recs(), inner)
        out[f"construct_{inner}_keys"] = np.array(list(rec))
        out[f"construct_{inner}_vals"] = np.stack([rec[k] for k in rec])
    msgs = []
    for args in t_rec.CHECK_ARGS:
        try:
            check_dynamic_rec_feats(*args)
            msgs.append("")
        except ValueError as e:
            msgs.append(str(e))
    out["check_messages"] = np.array(msgs)
    for strategy in ("average", "popular"):
        for inner_id in (True, False):
            ref = cold_start_rec(t_rec._cold_data_info(), t_rec.COLD_DEFAULT_RECS, strategy, t_rec.COLD_USERS, 6,
                                 inner_id)
            out[f"cold_{strategy}_{inner_id}"] = np.stack([ref[u] for u in t_rec.COLD_USERS])


def streams(out):
    for t, (uids, preds, K, N, consumed) in enumerate(t_rank.random_rank_cases()):
        out[f"rank_{t}"] = rank_recommendations("ranking", uids, preds, K, N, consumed, True, False, False)
    for t, (n_items, pos, num_neg) in enumerate(t_smp.random_negative_cases()):
        out[f"negatives_{t}"] = negatives_from_random(np.random.default_rng(t), n_items, pos, num_neg)


if __name__ == "__main__":
    out = {}
    di = feat_data_info()
    data_info_pieces(di, out)
    dynamic_rows(di, out)
    row_features("plain", di, out)
    row_features("multi_sparse", multi_sparse_data_info(), out)
    recommendation_shims(out)
    streams(out)
    np.savez_compressed(os.path.join(HERE, "reference_answers.npz"), **out)
    # a default_recs file exactly as the reference writes it (utils/save_load.py:39-42)
    save_default_recs(types.SimpleNamespace(default_recs=np.arange(2000)), HERE, "reference")
    print(sorted(out))
