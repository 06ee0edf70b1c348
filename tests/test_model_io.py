"""Model directory format: our writer's output reads back, and the same reader parses the
reference's own golden model (format fixture)."""
import os

import numpy as np
import pytest

import ydf_b200
from ydf_b200 import dataspec, model_io
from ydf_b200.model import GradientBoostedTreesModel

HERE = os.path.dirname(os.path.abspath(__file__))


def _toy_model(hessian=False, task="CLASSIFICATION"):
    cols = [dataspec.DiscretizedColumn("f0", np.array([-1.0, 0.0, 1.5], np.float32), 0.2, 4, 2),
            dataspec.DiscretizedColumn("f1", np.array([0.5], np.float32), 0.1, 2, 0)]
    spec = dataspec.DataSpec(columns=cols, label="y", task=task, label_classes=["a", "b"], num_rows=10)
    t = np.zeros(3, dtype=ydf_b200.NODE_DTYPE)
    t[0] = (1, 1, 0, 1, 1, 2, 0.25, 0.01, 10, 6, (1.5, 4.0, 10.0), 0, 0, (0,) * 8)
    t[1] = (-1, 0, 0, 2, -1, -1, 0.0, -0.2, 4, 0, (-2.0, 1.5, 4.0), 0, 0, (0,) * 8)
    t[2] = (-1, 0, 0, 2, -1, -1, 0.0, 0.3, 6, 0, (3.5, 2.5, 6.0), 0, 0, (0,) * 8)
    logs = [{"number_of_trees": 1, "loss": 1.1, "secondary": 0.7}]
    return GradientBoostedTreesModel(spec, [t], -0.4, "BINOMIAL_LOG_LIKELIHOOD" if task == "CLASSIFICATION"
                                     else "SQUARED_ERROR", logs, {"use_hessian_gain": int(hessian)})


@pytest.mark.parametrize("hessian", [False, True])
def test_write_and_read_back(tmp_path, hessian):
    m = _toy_model(hessian)
    p = str(tmp_path / "model")
    m.save(p)
    assert sorted(os.listdir(p)) == ["data_spec.pb", "done", "gradient_boosted_trees_header.pb", "header.pb",
                                     "nodes-00000-of-00001"]
    assert os.path.getsize(os.path.join(p, "done")) == 0
    r = model_io.read_ydf_model(p)
    assert r["name"] == "GRADIENT_BOOSTED_TREES" and r["task"] == 1 and r["label_col_idx"] == 0
    assert r["input_features"] == [1, 2] and r["num_trees"] == 1 and r["loss"] == 1
    assert r["node_format"] == "BLOB_SEQUENCE" and r["num_trees_per_iter"] == 1
    assert abs(r["initial_predictions"][0] + 0.4) < 1e-7
    n = r["nodes"]
    assert len(n) == 3
    assert n[0]["attribute"] == 2 and n[0]["discretized_threshold"] == 1 and n[0]["n_pos"] == 6
    assert n[0]["n"] == 10 and n[0]["n_cond"] == 10 and abs(n[0]["split_score"] - 0.25) < 1e-7
    assert "attribute" not in n[1] and abs(n[1]["top_value"] + 0.2) < 1e-7
    if hessian:
        assert n[2]["hessian_stats"] == (3.5, 2.5, 6.0)
    else:
        assert n[2]["distribution"] == (3.5, 2.5, 6.0)
    assert [c["name"] for c in r["columns"]] == ["y", "f0", "f1"]
    assert r["columns"][1]["type"] == 9  # DISCRETIZED_NUMERICAL
    np.testing.assert_array_equal(r["columns"][1]["boundaries"], np.array([-1.0, 0.0, 1.5], np.float32))
    assert r["created_num_rows"] == 10


def test_reader_parses_reference_format_fixture(tmp_path):
    """tests/golden/ydf_gbt_abalone_head.npz holds the files of the reference's golden model test_data/golden/gbt_abalone
    (file_<name>) and the head of that model as this reader decoded it (tests/golden/make_ydf_format_fixture.py).
    The files are decoded again and compared with the stored head."""
    fx = np.load(os.path.join(HERE, "golden", "ydf_gbt_abalone_head.npz"), allow_pickle=False)
    assert fx["node_format"] == "BLOB_SEQUENCE" and int(fx["num_trees"]) == 42 and int(fx["loss"]) == 2
    assert int(fx["root_n"]) == 1908 and int(fx["root_n_pos"]) == 1189
    # pre-order with the negative child first: node 1 holds the n - n_pos rows of the root
    assert int(fx["node1_n"]) == 1908 - 1189
    d = tmp_path / "gbt_abalone"
    d.mkdir()
    for k in fx.files:
        if k.startswith("file_"):
            (d / k[5:]).write_bytes(fx[k].tobytes())
    r = model_io.read_ydf_model(str(d))
    assert r["num_trees"] == 42 and r["nodes"][0]["n"] == 1908 and r["nodes"][0]["n_pos"] == 1189
    assert abs(r["nodes"][0]["higher_threshold"] - float(fx["root_threshold"])) == 0
    assert len(r["nodes"]) == int(fx["num_nodes"])
    assert r["initial_predictions"][0] == fx["initial_prediction"] and r["nodes"][0]["split_score"] == fx["root_score"]


def test_reference_golden_model_and_predictions(tmp_path):
    """Reads the reference's golden GBT model of Adult (68 trees with Higher and Contains{Vector,Bitmap} conditions;
    fixture tests/golden/ydf_adult_gbdt.npz = its files) and reproduces the golden predictions the reference's own
    `predict` tool wrote for adult_test (test_data/prediction/adult_test_binary_class_gbdt.csv).  Pins this repo's
    reading of the model format and of the condition semantics its writer emits: positive-set encodings, the
    pre-order node layout, NA handling through na_value, out-of-dictionary = 0."""
    import os
    G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    z = np.load(os.path.join(G, "ydf_adult_gbdt.npz"))
    d = tmp_path / "ref_model"
    d.mkdir()
    for k in z.files:
        if k.startswith("file_"):
            (d / k[5:]).write_bytes(z[k].tobytes())
    model = model_io.read_ydf_model(str(d))
    assert model["num_trees"] == 68 and model["loss"] == 1 and model["node_format"] == "BLOB_SEQUENCE"
    num, cat = np.load(os.path.join(G, "adult_numerical.npz")), np.load(os.path.join(G, "adult_categorical.npz"))
    cols = {}
    for c in ["age", "fnlwgt", "capital_gain", "capital_loss", "hours_per_week"]:
        cols[c] = num[f"test_{c}"].astype(np.float32)
    cols["education_num"] = num["test_education_num"].astype(str)       # CATEGORICAL in that model's dataspec
    for c in ["workclass", "education", "marital_status", "occupation", "relationship", "race", "sex", "native_country"]:
        cols[c] = cat[f"strings_{c}"][cat[f"test_{c}"]]
    raw = model_io.predict_ydf_model(model, cols)
    p = 1.0 / (1.0 + np.exp(-raw.astype(np.float64)))
    want = z["golden_p_positive"]
    assert len(p) == len(want) == 9769
    np.testing.assert_allclose(p, want, rtol=0, atol=2e-6)               # the CSV holds 6 significant digits
    acc = np.mean((p > 0.5) == (num["test_income"] == 1))
    assert 0.86 < acc < 0.88
    # the encoding rule of categorical conditions (learner/decision_tree/utils.cc:31-63) as the reference applied it:
    # a bitmap of ceil(K / 8) bytes whenever that is not larger than 4 bytes per positive category
    n_bitmap = 0
    for rec in model_io.read_blob_sequence(str(d / "nodes-00000-of-00001")):
        cond = model_io._one(model_io.pb_decode(rec), 3)
        if cond is None:
            continue
        c = model_io.pb_decode(cond)
        K = model["columns"][model_io._one(c, 2)].get("number_of_unique_values")
        for ff, _, v in model_io.pb_decode(model_io._one(c, 3)):
            if ff == 5:
                bm = model_io._one(model_io.pb_decode(v), 1, b"")
                assert len(bm) == (K + 7) // 8 and (K + 7) // 8 <= 4 * sum(bin(b).count("1") for b in bm)
                n_bitmap += 1
            elif ff == 4:
                packed = model_io._one(model_io.pb_decode(v), 1, b"")
                assert (K + 7) // 8 > 4 * sum(1 for b in packed if not b & 0x80)
    assert n_bitmap == 1100


def test_written_model_evaluates_like_the_python_mirror(tmp_path):
    """Writer -> reader -> generic evaluation (the one pinned by the reference's golden predictions above) agrees with
    GradientBoostedTreesModel.predict on a model with DiscretizedHigher and Contains conditions and missing values."""
    from ydf_b200 import dataspec
    num = dataspec.DiscretizedColumn("x", np.array([-0.5, 0.25, 1.5], np.float32), 0.1, 4, 1)
    cat = dataspec.CategoricalColumn("c", ["<OOD>", "u", "v", "w"], [0, 9, 7, 5], 4, 1)
    spec = dataspec.DataSpec(columns=[num, cat], label="y", task="REGRESSION", num_rows=10)
    t = np.zeros(5, dtype=ydf_b200.NODE_DTYPE)
    # pre-order (node, negative subtree, positive subtree), the layout the engine emits and the format stores
    t[0] = (0, 2, 0, 1, 1, 4, 0.5, 0.0, 10, 4, (0, 0, 10), 0, 0, (0,) * 8)            # x bin >= 2 (NA -> bin 1 -> negative)
    t[1] = (1, 0, 1, 2, 2, 3, 0.2, 0.0, 6, 3, (0, 0, 6), 1, 0, (0b0110,) + (0,) * 7)   # c in {u, v}; NA -> u -> positive
    t[2] = (-1, 0, 0, 3, -1, -1, 0, -0.4, 3, 0, (0, 0, 3), 0, 0, (0,) * 8)
    t[3] = (-1, 0, 0, 3, -1, -1, 0, 0.1, 3, 0, (0, 0, 3), 0, 0, (0,) * 8)
    t[4] = (-1, 0, 0, 2, -1, -1, 0, 0.7, 4, 0, (0, 0, 4), 0, 0, (0,) * 8)
    model = ydf_b200.GradientBoostedTreesModel(spec, [t, t], 0.25, "SQUARED_ERROR")
    model.save(str(tmp_path / "m"))
    back = model_io.read_ydf_model(str(tmp_path / "m"))
    data = {"x": np.array([-1.0, 0.3, 2.0, np.nan, 0.0, 9.0], np.float32),
            "c": np.array(["u", "w", "v", "", "zzz", "w"], dtype=object)}
    want = model.predict(data)
    got = model_io.predict_ydf_model(back, data)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-7)
    np.testing.assert_allclose(want, 0.25 + 2 * np.array([0.1, 0.7, 0.7, 0.1, -0.4, 0.7], np.float32), atol=1e-6)
