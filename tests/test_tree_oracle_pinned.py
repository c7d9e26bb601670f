"""Pins oracle/tree_oracle.c (+ the boosting restatement in oracle/tree.py) against trees grown by the unmodified
reference library: the committed golden files (tests/golden/tree_golden.json, and a further run in tests/golden/reference_golden.json).
Integer-valued features are used so that the reference's bins are known without restating its bin finder: value k sits
in bin k (BinMapper::FindBin with <= max_bin distinct values; GreedyFindBin bin.cpp:83-98 puts bounds at midpoints)."""
import json
import os

import numpy as np
import pytest

import treedata
from oracle import tree as ot

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIVE_SPEC = {"name": "live", "n": 3000, "F": 5, "kind": "int", "levels": 60, "num_leaves": 12, "min_data_in_leaf": 15, "num_iter": 2, "seed": 11}


@pytest.fixture(scope="module")
def tree_golden():
    with open(os.path.join(ROOT, "tests", "golden", "tree_golden.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def golden_ref():
    with open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")) as f:
        return json.load(f)


def _cfg(spec):
    return ot.make_config(num_leaves=spec["num_leaves"], min_data_in_leaf=spec["min_data_in_leaf"], lambda_l2=spec.get("lambda_l2", 0.),
                          min_gain_to_split=spec.get("min_gain_to_split", 0.), max_depth=spec.get("max_depth", -1))


def _check(otrees, gtrees, init, leaf_tol):
    assert len(otrees) == len(gtrees)
    for k, (a, g) in enumerate(zip(otrees, gtrees)):
        assert a["num_leaves"] == g["num_leaves"]
        assert np.array_equal(a["split_feature"], np.array(g["split_feature"]))
        assert np.array_equal(a["threshold_bin"], np.floor(np.array(g["threshold"])).astype(int))
        assert np.array_equal(a["left_child"], np.array(g["left_child"])) and np.array_equal(a["right_child"], np.array(g["right_child"]))
        assert np.array_equal(a["leaf_count"], np.array(g["leaf_count"]))
        lv = a["leaf_value"] + (init if k == 0 else 0.)
        assert np.max(np.abs(lv - np.array(g["leaf_value"]))) <= leaf_tol * np.max(np.abs(g["leaf_value"]))


def test_tree_oracle_matches_reference_golden(tree_golden):
    for rec in tree_golden["cases"]:
        spec = rec["spec"]
        if spec["kind"] != "int":
            continue
        X, y, _ = treedata.make_case(spec)
        bins = np.ascontiguousarray(X.T.astype(np.uint8))
        trees, score, init = ot.boost_l2(bins, np.full(spec["F"], spec["levels"]), y, _cfg(spec), 0.1, spec["num_iter"])
        _check(trees, rec["trees"], init, 1e-15)  # same summation order as the reference's column-wise path: bit-exact
        assert np.abs(score[:64] - np.array(rec["score_head"])).max() == 0.0


def test_tree_oracle_matches_reference_live(golden_ref):
    from gpboost_b200.booster import parse_model_string
    spec = LIVE_SPEC
    X, y, _ = treedata.make_case(spec)
    rec = golden_ref["tree"]
    g = parse_model_string(rec["model"])
    bins = np.ascontiguousarray(X.T.astype(np.uint8))
    trees, score, init = ot.boost_l2(bins, np.full(spec["F"], spec["levels"]), y, _cfg(spec), 0.1, spec["num_iter"])
    _check(trees, [{k: v for k, v in t.items()} for t in g], init, 1e-15)
    assert np.abs(score - np.array(rec["score"])).max() == 0.0
