"""Generates tests/golden/reference_golden.json: what the UNMODIFIED reference library (oracle/_ref/lib_gpboost.so, built by
oracle/Makefile.ref) returns for the comparisons of test_oracle_pinned, test_tree_oracle_pinned, test_vecchia_gpu, test_model_text_io
and test_dropin_reference_package, so that those tests compare with the reference without needing it at run time. The drop-in
section runs the reference's own Python package (from the same reference checkout, oracle.build.REFERENCE_DIR) on that library:
    python tests/golden/make_reference_golden.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import datagen  # noqa: E402
import dropin  # noqa: E402
import test_dropin_reference_package as tdr  # noqa: E402
import test_model_text_io as tio  # noqa: E402
import test_oracle_pinned as top  # noqa: E402
import test_tree_oracle_pinned as ttp  # noqa: E402
import test_vecchia_gpu as tvg  # noqa: E402
import treedata  # noqa: E402
from gpboost_b200 import GPModel  # noqa: E402
from gpboost_b200.booster import Booster, Dataset, parse_model_string  # noqa: E402
from gpboost_b200.libpath import load_lib  # noqa: E402
from oracle import ref_lib_path  # noqa: E402

assert dropin.ref_package_dir() is not None, "no reference checkout: set GPBOOST_REFERENCE"
ref = load_lib(ref_lib_path())
out = {"generator": "tests/golden/make_reference_golden.py", "reference": "fabsig/GPBoost c93fa49 (v1.7.3), CPU build"}

# test_oracle_pinned: Vecchia likelihoods of the three live cases
coords, y = datagen.synth(1200, 2, 21)
out["vecchia_nll"] = []
for cov, shape, m, ordering in top.LIVE_CASES:
    mdl = GPModel(gp_coords=coords, cov_function=cov, cov_fct_shape=shape, gp_approx="vecchia", num_neighbors=m,
                  vecchia_ordering=ordering, seed=4, _lib=ref)
    out["vecchia_nll"].append({"cov_function": cov, "cov_fct_shape": shape, "num_neighbors": m, "vecchia_ordering": ordering,
                               "negll": mdl.neg_log_likelihood(top.LIVE_CP, y)})

# test_tree_oracle_pinned: two boosting iterations on integer features
spec = ttp.LIVE_SPEC
X, y, _ = treedata.make_case(spec)
params = treedata.booster_params(spec, reference=True)
b = Booster(params, Dataset(X, y, params=params, _lib=ref), _lib=ref)
for _ in range(spec["num_iter"]):
    b.update()
out["tree"] = {"model": b.model_to_string(), "score": b.inner_predict_train().tolist()}

# test_vecchia_gpu: likelihood at fixed parameters and at the fitted optimum
coords, y = datagen.synth(2500, 2, 29)
mdl = GPModel(gp_coords=coords, _lib=ref, **tvg.LIVE_KW)
out["vecchia_capi"] = {"negll": mdl.neg_log_likelihood(tvg.LIVE_CP, y)}
mdl.fit(y)
out["vecchia_capi"]["fit_negll"] = mdl.get_current_neg_log_likelihood()

# test_model_text_io: a model trained by the reference, its predictions, importances and iteration ranges
X, y = tio.train_data()
params = tio.PARAMS
b = Booster(params, Dataset(X, y, params=params, _lib=ref), _lib=ref)
for _ in range(12):
    b.update()
Xt = tio.predict_data()
rec = {"model": b.model_to_string(), "pred": b.predict(Xt).tolist(), "ranges": [], "feature_importance": []}
for st, nit in tio.RANGES:
    rec["ranges"].append({"start_iteration": st, "num_iteration": nit, "pred": b.predict(Xt, start_iteration=st, num_iteration=nit).tolist(),
                          "leaf_value": [t["leaf_value"].tolist() for t in parse_model_string(b.model_to_string(st, nit))]})
for typ in (0, 1):
    for nit in (-1, 5):
        v = np.zeros(6)
        assert ref.LGBM_BoosterFeatureImportance(b.handle, nit, typ, v.ctypes.data_as(tio.C.POINTER(tio.C.c_double))) == 0
        rec["feature_importance"].append({"importance_type": typ, "num_iteration": nit, "values": v.tolist()})
lv = tio.C.c_double(0.)
assert ref.LGBM_BoosterGetLeafValue(b.handle, 3, 2, tio.C.byref(lv)) == 0
rec["leaf_value_3_2"] = lv.value
out["model_text_io"] = rec

# test_model_text_io: models trained on data with NaNs and with zero_as_missing
y, train_sets, Xt = tio.missing_value_data()
out["missing_values"] = []
for Xtr, extra in train_sets:
    params = dict(tio.MISSING_PARAMS, **extra)
    b = Booster(params, Dataset(Xtr, y, params=params, _lib=ref), _lib=ref)
    for _ in range(8):
        b.update()
    out["missing_values"].append({"params": extra, "model": b.model_to_string(), "pred": b.predict(Xt).tolist()})

# test_dropin_reference_package: the drop-in script, run by the reference's package on the reference library
out["dropin"] = dropin.run_with(ref_lib_path(), tdr.SCRIPT)

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_golden.json"), "w") as f:
    json.dump(out, f)
