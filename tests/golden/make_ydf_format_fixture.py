"""Generates tests/golden/ydf_gbt_abalone_head.npz from the reference's golden model: the files of
test_data/golden/gbt_abalone (as file_<name> byte arrays) and what this reader decodes from them.
usage: make_ydf_format_fixture.py <reference checkout>/yggdrasil_decision_forests/test_data/golden/gbt_abalone"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import ydf_b200  # noqa: E402
from ydf_b200 import model_io  # noqa: E402

src = sys.argv[1]
files = {"file_" + f: np.frombuffer(open(os.path.join(src, f), "rb").read(), dtype=np.uint8)
         for f in sorted(os.listdir(src))}
r = model_io.read_ydf_model(src)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ydf_gbt_abalone_head.npz"),
                    node_format=r["node_format"], num_trees=r["num_trees"], loss=r["loss"],
                    initial_prediction=r["initial_predictions"][0], num_nodes=len(r["nodes"]),
                    root_n=r["nodes"][0]["n"], root_n_pos=r["nodes"][0]["n_pos"],
                    root_threshold=r["nodes"][0]["higher_threshold"], root_score=r["nodes"][0]["split_score"],
                    node1_n=r["nodes"][1]["n"], **files)
print("ok", len(r["nodes"]))
