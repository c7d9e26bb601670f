"""Model text I/O of the boosting side (LGBM_BoosterSaveModelToString / SaveModel / LoadModelFromString / CreateFromModelfile /
PredictForMat; gbdt_model_text.cpp, tree.cpp) — host logic, no device needed, checked against the unmodified reference library
through its stored results (tests/golden/reference_golden.json, tests/golden/make_reference_golden.py):
  * a model trained by the REFERENCE is loaded by the B200 library: identical raw predictions (host tree traversal);
  * the B200 library's writer output (of that loaded model) carries the reference's trees and, where the reference library is
    built, is loaded back by the REFERENCE with identical predictions — the text this build writes carries every field the
    reference's loader insists on (feature_names, feature_infos, …);
  * file round trip through LGBM_BoosterSaveModel / LGBM_BoosterCreateFromModelfile."""
import ctypes as C
import json
import os
import tempfile

import numpy as np
import pytest

from gpboost_b200.booster import Booster, Dataset, parse_model_string
from gpboost_b200.libpath import load_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = dict(objective="regression", num_leaves=15, min_data_in_leaf=20, learning_rate=0.1, max_bin=255, verbose=-1)
MISSING_PARAMS = dict(objective="regression", num_leaves=15, min_data_in_leaf=20, learning_rate=0.1, verbose=-1)
RANGES = ((0, 5), (3, 4), (10, 50), (0, -1), (12, 3))


def train_data():
    rng = np.random.default_rng(0)
    X = rng.random((2000, 6)); X[:, 4] = 3.0  # one constant (trivial) feature
    X[:, 5] = np.round(X[:, 5] * 4) - 2.        # few distinct values incl. negatives and zero
    y = np.sin(3 * X[:, 0]) + X[:, 1] ** 2 + 0.3 * X[:, 5] + 0.1 * rng.standard_normal(2000)
    return X, y


def predict_data():
    Xt = np.random.default_rng(1).random((500, 6)) * 1.2 - 0.1
    Xt[:, 5] = np.round(Xt[:, 5] * 4) - 2.
    return Xt


def missing_value_data():
    """Training targets, [(training matrix with NaNs, {}), (training matrix with zeros, {"zero_as_missing": True})], test matrix."""
    rng = np.random.default_rng(5)
    X = rng.standard_normal((3000, 4)); y = X[:, 0] + (X[:, 1] > 0) + 0.1 * rng.standard_normal(3000)
    Xn = X.copy(); Xn[rng.random(X.shape) < 0.15] = np.nan
    Xz = X.copy(); Xz[rng.random(X.shape) < 0.3] = 0.
    Xt = rng.standard_normal((400, 4)); Xt[rng.random(Xt.shape) < 0.2] = np.nan; Xt[rng.random(Xt.shape) < 0.2] = 0.
    return y, [(Xn, {}), (Xz, {"zero_as_missing": True})], Xt


@pytest.fixture(scope="module")
def golden_ref():
    with open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def ref_model(golden_ref):
    """(reference model text, test matrix, the reference's predictions on it, the rest of the stored record)"""
    rec = golden_ref["model_text_io"]
    return rec["model"], predict_data(), np.array(rec["pred"]), rec


def test_reference_model_loads_and_predicts_identically(ref_model, product_lib):
    text, Xt, want, _ = ref_model
    ours = Booster(model_str=text, _lib=product_lib)
    assert ours.current_iteration() == 12
    assert np.array_equal(ours.predict(Xt), want)


def test_writer_output_is_loadable_by_the_reference(ref_model, product_lib, ref_lib):
    text, Xt, want, _ = ref_model
    ours = Booster(model_str=text, _lib=product_lib)
    text2 = ours.model_to_string()
    if ref_lib is not None:
        back = Booster(model_str=text2, _lib=ref_lib)  # the reference's loader on OUR text
        assert np.array_equal(back.predict(Xt), want)
    assert np.array_equal(Booster(model_str=text2, _lib=product_lib).predict(Xt), want)
    a, b = parse_model_string(text), parse_model_string(text2)
    assert len(a) == len(b) == 12
    for ta, tb in zip(a, b):
        for k in ("split_feature", "left_child", "right_child", "leaf_count"):
            assert np.array_equal(ta[k], tb[k]), k
        assert np.array_equal(ta["threshold"], tb["threshold"]) and np.array_equal(ta["leaf_value"], tb["leaf_value"])


def test_file_round_trip(ref_model, product_lib):
    text, Xt, want, _ = ref_model
    ours = Booster(model_str=text, _lib=product_lib)
    with tempfile.TemporaryDirectory() as d:
        fn = os.path.join(d, "model.txt")
        ours.save_model(fn)
        again = Booster(model_file=fn, _lib=product_lib)
        assert np.array_equal(again.predict(Xt), want)


def test_load_errors_use_the_error_channel(product_lib):
    from gpboost_b200.basic import GPBoostError
    with pytest.raises(GPBoostError):
        Booster(model_str="tree\nversion=v3\nnum_class=1\n", _lib=product_lib)
    with pytest.raises(GPBoostError):
        Booster(model_file="/nonexistent/model.txt", _lib=product_lib)


def test_feature_importance_and_leaf_values_match_the_reference(ref_model, product_lib):
    text, _, _, rec = ref_model
    ours = Booster(model_str=text, _lib=product_lib)
    assert len(rec["feature_importance"]) == 4
    for fi in rec["feature_importance"]:
        typ, nit, b = fi["importance_type"], fi["num_iteration"], np.array(fi["values"])
        a = np.zeros(6)
        assert product_lib.LGBM_BoosterFeatureImportance(ours.handle, nit, typ, a.ctypes.data_as(C.POINTER(C.c_double))) == 0
        assert np.allclose(a, b, rtol=1e-6, atol=0), (typ, nit, a, b)  # gains are printed with 6 significant digits in the text
    va = C.c_double(0.)
    assert product_lib.LGBM_BoosterGetLeafValue(ours.handle, 3, 2, C.byref(va)) == 0
    assert va.value == rec["leaf_value_3_2"]


def test_iteration_ranges_of_predict_and_save_match_the_reference(ref_model, product_lib):
    """start_iteration / num_iteration of LGBM_BoosterPredictForMat and LGBM_BoosterSaveModelToString (c_api.h:1020, :1200)."""
    text, Xt, _, rec = ref_model
    ours = Booster(model_str=text, _lib=product_lib)
    assert [(r["start_iteration"], r["num_iteration"]) for r in rec["ranges"]] == list(RANGES)
    for r in rec["ranges"]:
        st, nit = r["start_iteration"], r["num_iteration"]
        assert np.array_equal(ours.predict(Xt, start_iteration=st, num_iteration=nit), np.array(r["pred"])), (st, nit)
        a = parse_model_string(ours.model_to_string(st, nit))
        assert len(a) == len(r["leaf_value"]), (st, nit)
        for ta, lv in zip(a, r["leaf_value"]):
            assert np.array_equal(ta["leaf_value"], np.array(lv))


def test_missing_value_routing_of_a_reference_model(golden_ref, product_lib):
    """A reference model trained on data with NaNs (decision_type 8 / 10: MissingType::NaN) and one with zero_as_missing
    (decision_type 4 / 6) route NaN / zero inputs like the reference's NumericalDecision (tree.h:329-347)."""
    _, train_sets, Xt = missing_value_data()
    recs = golden_ref["missing_values"]
    assert [r["params"] for r in recs] == [extra for _, extra in train_sets]
    seen = set()
    for r in recs:
        text = r["model"]
        for line in text.split("\n"):
            if line.startswith("decision_type="):
                seen.update(int(v) for v in line.split("=")[1].split())
        ours = Booster(model_str=text, _lib=product_lib)
        assert np.array_equal(ours.predict(Xt), np.array(r["pred"]))
        assert np.array_equal(parse_model_string(ours.model_to_string())[0]["leaf_value"], parse_model_string(text)[0]["leaf_value"])
        assert "decision_type=" + text.split("decision_type=")[1].split("\n")[0] in ours.model_to_string()
    assert seen & {8, 10} and seen & {4, 6}, seen


def test_corrupt_models_and_unsupported_parameters_fail_cleanly(ref_model, product_lib):
    from gpboost_b200.basic import GPBoostError
    text = ref_model[0]
    lines = text.split("\n")
    def mutate(key, fn):
        out, done = [], False
        for ln in lines:
            if not done and ln.startswith(key + "="):
                vals = ln.split("=")[1].split(); ln = key + "=" + " ".join(fn(vals)); done = True
            out.append(ln)
        return "\n".join(out)
    for bad in (mutate("split_feature", lambda v: ["999"] + v[1:]), mutate("left_child", lambda v: ["0"] + v[1:]),
                mutate("right_child", lambda v: v[:-1] + ["-500"]), mutate("left_child", lambda v: v[:1] + ["1"] + v[2:])):
        with pytest.raises(GPBoostError):
            Booster(model_str=bad, _lib=product_lib)
    X = np.random.default_rng(0).random((200, 3))
    for p in ({"subsample": 0.5}, {"colsample_bytree": 0.5}, {"boosting": "dart"}, {"reg_alpha": 0.1}, {"max_delta_step": 1.0},
              {"linear_tree": True}, {"categorical_feature": "0,1"}, {"monotone_constraints": "1,0,0"}, {"extra_trees": True}):
        with pytest.raises(GPBoostError) as e:
            Dataset(X, X[:, 0], params=dict(p, verbose=-1), _lib=product_lib)
        assert "not supported by the B200 build" in str(e.value), p
