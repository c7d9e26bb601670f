"""Drop-in proof (SURVEY §8b): the UNMODIFIED reference Python package drives the product library on the device —
gpb.GPModel(...).fit(y), neg_log_likelihood, gpb.train(params, ds, gp_model=...) — and the results are compared with what the same
script gives on the unmodified reference library (stored in tests/golden/reference_golden.json by
tests/golden/make_reference_golden.py). The package is not part of this repository, so where it is absent the same workload runs
through this repository's own frontend (gpboost_b200.GPModel / Booster) against the same stored results.
CPU part: the script itself runs on the reference library."""
import json
import os

import numpy as np
import pytest

import dropin

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRODUCT = os.path.join(ROOT, "gpboost_b200", "lib_gpboost_b200.so")

SCRIPT = """
rng = np.random.default_rng(7)
n = 600
coords = rng.random((n, 2))
X = rng.random((n, 3))
f = np.sin(4 * coords[:, 0]) + np.cos(3 * coords[:, 1])
y = f + 0.3 * rng.standard_normal(n)
# ---- GPModel: fit, likelihood
m = gpb.GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=10,
                vecchia_ordering="random", seed=1)
m.fit(y=y)
out["cov_pars"] = np.asarray(m.get_cov_pars()).reshape(-1).tolist()
out["num_it"] = int(m._get_num_optim_iter()) if hasattr(m, "_get_num_optim_iter") else -1
out["negll_at"] = float(m.neg_log_likelihood(cov_pars=np.array([0.3, 1.0, 0.2]), y=y))
out["negll_opt"] = float(m.get_current_neg_log_likelihood())
# ---- grouped random effect
g = rng.integers(0, 40, n)
yg = 0.7 * rng.standard_normal(40)[g] + 0.5 * rng.standard_normal(n)
mg = gpb.GPModel(group_data=g)
mg.fit(y=yg)
out["cov_pars_grouped"] = np.asarray(mg.get_cov_pars()).reshape(-1).tolist()
# ---- GPBoost: trees + GP
m2 = gpb.GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=10,
                 vecchia_ordering="random", seed=1)
yb = 2 * np.sin(3 * X[:, 0]) + X[:, 1] ** 2 + f + 0.2 * rng.standard_normal(n)
ds = gpb.Dataset(X, yb)
params = {"objective": "regression_l2", "learning_rate": 0.1, "num_leaves": 8, "min_data_in_leaf": 20, "verbose": -1}
bst = gpb.train(params=params, train_set=ds, gp_model=m2, num_boost_round=6)
out["cov_pars_boost"] = np.asarray(m2.get_cov_pars()).reshape(-1).tolist()
txt = bst.model_to_string()
if txt.lstrip().startswith("{"):   # with a GP model the package wraps the tree model text and the GPModel's state in JSON
    txt = json.loads(txt)["booster_str"]
out["num_trees"] = bst.num_trees()
out["split_feature"] = [ln for ln in txt.split("\\n") if ln.startswith("split_feature=")]
out["threshold"] = [ln for ln in txt.split("\\n") if ln.startswith("threshold=")]
out["leaf_count"] = [ln for ln in txt.split("\\n") if ln.startswith("leaf_count=")]
# ---- plain boosting, tree predictions on new data
ds2 = gpb.Dataset(X, yb)
bst2 = gpb.train(params=params, train_set=ds2, num_boost_round=5)
out["pred"] = bst2.predict(rng.random((20, 3))).tolist()
"""


def run_frontend(lib=None):
    """SCRIPT through gpboost_b200's frontend (`lib`: the library to bind, default the product library); same outputs."""
    from gpboost_b200 import GPModel
    from gpboost_b200.booster import Booster, Dataset, parse_model_string
    out = {}
    rng = np.random.default_rng(7)
    n = 600
    coords = rng.random((n, 2))
    X = rng.random((n, 3))
    f = np.sin(4 * coords[:, 0]) + np.cos(3 * coords[:, 1])
    y = f + 0.3 * rng.standard_normal(n)
    m = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=10,
                vecchia_ordering="random", seed=1, _lib=lib)
    m.fit(y=y)
    out["cov_pars"] = m.get_cov_pars().tolist()
    out["num_it"] = m._get_num_optim_iter()
    out["negll_at"] = m.neg_log_likelihood(cov_pars=np.array([0.3, 1.0, 0.2]), y=y)
    out["negll_opt"] = m.get_current_neg_log_likelihood()
    g = rng.integers(0, 40, n)
    yg = 0.7 * rng.standard_normal(40)[g] + 0.5 * rng.standard_normal(n)
    mg = GPModel(group_data=g, _lib=lib)
    mg.fit(y=yg)
    out["cov_pars_grouped"] = mg.get_cov_pars().tolist()
    m2 = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=10,
                 vecchia_ordering="random", seed=1, _lib=lib)
    yb = 2 * np.sin(3 * X[:, 0]) + X[:, 1] ** 2 + f + 0.2 * rng.standard_normal(n)
    params = {"objective": "regression_l2", "learning_rate": 0.1, "num_leaves": 8, "min_data_in_leaf": 20, "verbose": -1}
    # gpb.train(..., gp_model=...) adds these two (engine.py of the package)
    gp_params = dict(params, use_gp_model_for_validation=True, train_gp_model_cov_pars=True)
    bst = Booster(gp_params, Dataset(X, yb, params=gp_params, _lib=lib), gp_model=m2, _lib=lib)
    for _ in range(6):
        bst.update()
    out["cov_pars_boost"] = m2.get_cov_pars().tolist()
    txt = bst.model_to_string()
    out["num_trees"] = len(parse_model_string(txt))
    out["split_feature"] = [ln for ln in txt.split("\n") if ln.startswith("split_feature=")]
    out["threshold"] = [ln for ln in txt.split("\n") if ln.startswith("threshold=")]
    out["leaf_count"] = [ln for ln in txt.split("\n") if ln.startswith("leaf_count=")]
    bst2 = Booster(params, Dataset(X, yb, params=params, _lib=lib), _lib=lib)
    for _ in range(5):
        bst2.update()
    out["pred"] = bst2.predict(rng.random((20, 3))).tolist()
    return out


def golden_dropin():
    with open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")) as f:
        return json.load(f)["dropin"]


def check_against_reference(got, want):
    # fits: the two optimisers agree on the optimum to the reference's own convergence tolerance (relative NLL change 1e-6)
    assert np.allclose(got["cov_pars"], want["cov_pars"], rtol=2e-3), (got["cov_pars"], want["cov_pars"])
    assert abs(got["negll_opt"] - want["negll_opt"]) <= 1e-5 * abs(want["negll_opt"])
    assert abs(got["negll_at"] - want["negll_at"]) <= 1e-8 * abs(want["negll_at"])
    assert np.allclose(got["cov_pars_grouped"], want["cov_pars_grouped"], rtol=2e-3)
    # GPBoost: same trees (integer decisions bit-exact), covariance parameters to the fit tolerance
    assert got["num_trees"] == want["num_trees"]
    assert got["split_feature"][0] == want["split_feature"][0] and got["threshold"][0] == want["threshold"][0]
    assert got["leaf_count"][0] == want["leaf_count"][0]
    assert np.allclose(got["cov_pars_boost"], want["cov_pars_boost"], rtol=5e-3)
    assert np.allclose(got["pred"], want["pred"], rtol=1e-10, atol=1e-12)


def _ref_lib_path():
    from oracle import ref_lib_path
    p = ref_lib_path()
    return p if os.path.exists(p) else None


@pytest.mark.skipif(dropin.ref_package_dir() is None, reason="reference Python package not present")
def test_script_runs_on_the_reference_library():
    ref = _ref_lib_path()
    if ref is None:
        pytest.skip("reference library not built")
    r = dropin.run_with(ref, SCRIPT)
    assert r["num_trees"] == 6 and len(r["cov_pars"]) == 3 and len(r["pred"]) == 20


@pytest.mark.gpu
@pytest.mark.skipif(dropin.ref_package_dir() is None, reason="reference Python package not present (set GPBOOST_REFERENCE)")
def test_unmodified_package_on_the_device_matches_the_reference_library():
    check_against_reference(dropin.run_with(PRODUCT, SCRIPT), golden_dropin())


@pytest.mark.gpu
def test_frontend_on_the_device_matches_the_reference_library():
    check_against_reference(run_frontend(), golden_dropin())
