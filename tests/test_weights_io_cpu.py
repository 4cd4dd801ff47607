"""Round trips through the reference's on-disk weight formats (utils/save_load.py:39-98,
bases/embed_base.py:289-330); the reference's own default_recs file (tests/golden/reference_default_recs.npz,
written by tests/golden/gen_reference_answers.py) pins that format."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_embed_and_tf_variable_roundtrip(tmp_path):
    from librecommender_b200 import weights_io as io

    rng = np.random.default_rng(0)
    U, I = rng.standard_normal((11, 8)).astype(np.float32), rng.standard_normal((7, 8)).astype(np.float32)
    io.save_embed_model(str(tmp_path), "m", U, I)
    u2, i2 = io.load_embed_model(str(tmp_path), "m")
    np.testing.assert_array_equal(u2, U)
    np.testing.assert_array_equal(i2, I)
    raw = np.load(os.path.join(tmp_path, "m.npz"))
    assert set(raw.files) == {"user_embed", "item_embed"}            # the keys EmbedBase.load reads

    w = dict(user_embeds=U, item_embeds=I, sparse_embeds=rng.standard_normal((30, 8)).astype(np.float32),
             user_linear=rng.standard_normal(11).astype(np.float32), item_linear=rng.standard_normal(7).astype(np.float32),
             sparse_linear=rng.standard_normal(30).astype(np.float32), lin_kernel=rng.standard_normal(5).astype(np.float32))
    io.save_tf_variables(str(tmp_path), "fm", w, extra_names={"lin_kernel": "dense/kernel:0"})
    raw = np.load(os.path.join(tmp_path, "fm_tf_variables.npz"))
    # shapes = the reference's var_shape values (fm.py:181-249): id tables [V, 1], feature tables 1-D
    assert raw["embedding/user_linear_var:0"].shape == (11, 1)
    assert raw["embedding/item_linear_var:0"].shape == (7, 1)
    assert raw["embedding/sparse_linear_var:0"].shape == (30,)
    back = io.load_tf_variables(str(tmp_path), "fm", extra_names={"lin_kernel": "dense/kernel:0"})
    for k in w:
        np.testing.assert_array_equal(np.asarray(back[k]).reshape(w[k].shape), w[k])
    io.save_default_recs(str(tmp_path), "m", np.arange(20))
    np.testing.assert_array_equal(io.load_default_recs(str(tmp_path), "m"), np.arange(20))


def test_reference_loader_reads_our_default_recs(tmp_path):
    """Our file has the layout of the reference's (utils/save_load.py:39-48 reads key "default_recs" of
    ``<name>_default_recs.npz``), and our loader reads the reference's file."""
    from librecommender_b200 import weights_io as io

    io.save_default_recs(str(tmp_path), "m", np.arange(2000))
    ours = np.load(os.path.join(tmp_path, "m_default_recs.npz"))
    ref = np.load(os.path.join(GOLDEN, "reference_default_recs.npz"))
    assert ours.files == ref.files
    assert ours["default_recs"].dtype == ref["default_recs"].dtype
    np.testing.assert_array_equal(ours["default_recs"], ref["default_recs"])
    np.testing.assert_array_equal(io.load_default_recs(GOLDEN, "reference"), np.arange(2000))


@pytest.mark.parametrize("arch,n_hidden,use_bn", [("FM", 0, True), ("DeepFM", 3, True), ("DeepFM", 2, False),
                                                   ("DIN", 3, True), ("YouTubeRanking", 2, True), ("TwoTower", 2, True)])
def test_auto_named_tf_variables_resolve_without_hand_written_map(tmp_path, arch, n_hidden, use_bn):
    """A ``*_tf_variables.npz`` laid out with TensorFlow's creation-order names loads into the engine
    weight structure with no name map from the caller; a missing variable is reported by name."""
    from librecommender_b200 import weights_io as io

    rng = np.random.default_rng(0)
    names = io.default_tf_names(arch, n_hidden, use_bn)
    flat = {}

    def fill(n):
        if isinstance(n, dict):
            return {k: fill(v) for k, v in n.items()}
        if isinstance(n, list):
            return [fill(v) for v in n]
        flat[n] = rng.standard_normal((3, 2)).astype(np.float32)
        return flat[n]

    expect = fill(names)
    assert len(set(flat)) == len(flat)                                   # every variable has its own name
    flat["embedding/user_embeds_var:0"] = rng.standard_normal((5, 4)).astype(np.float32)
    flat["embedding/item_embeds_var:0"] = rng.standard_normal((6, 4)).astype(np.float32)
    np.savez(os.path.join(tmp_path, "m_tf_variables.npz"), **flat)
    w = io.load_reference_tf_model(str(tmp_path), "m", arch, n_hidden, use_bn)

    def same(a, b):
        if isinstance(a, dict):
            assert set(a) == set(b)
            for k in a:
                same(a[k], b[k])
        elif isinstance(a, list):
            assert len(a) == len(b)
            for x, y in zip(a, b):
                same(x, y)
        else:
            np.testing.assert_array_equal(a, b)

    for k in names:
        same(expect[k], w[k])
    np.testing.assert_array_equal(w["user_embeds"], flat["embedding/user_embeds_var:0"])
    # the name table follows the creation order of the reference's graph builders
    if arch == "DeepFM" and use_bn:
        assert names["mlp"]["bn_in"]["gamma"] == "mlp/batch_normalization/gamma:0"
        assert names["mlp"]["kernels"][1] == "mlp/mlp_layer2/kernel:0"
        assert names["mlp"]["bns"][0]["mean"] == "mlp/batch_normalization_1/moving_mean:0"
        assert names["out_kernel"] == "dense_1/kernel:0" and names["lin_kernel"] == "dense/kernel:0"
    some = next(n for n in flat if not n.startswith("embedding/"))
    del flat[some]
    np.savez(os.path.join(tmp_path, "bad_tf_variables.npz"), **flat)
    with pytest.raises(KeyError, match=some.replace("/", "/")):
        io.load_reference_tf_model(str(tmp_path), "bad", arch, n_hidden, use_bn)
