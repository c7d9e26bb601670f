"""The oracle (oracle/vecchia_oracle.c) is pinned against (1) the known-answer values hard-coded in the
reference's own R tests, (2) golden vectors produced by the unmodified reference library
(tests/golden/make_golden.py) and (3) the results of calls of that library on further cases (tests/golden/make_reference_golden.py)."""
import json
import os

import numpy as np
import pytest

import datagen
from conftest import case_data
from oracle import vecchia as ov

CP = np.array([0.1, 1.6, 0.2])
LIVE_CASES = (("matern", 1.5, 15, "random"), ("exponential", 0.5, 8, "none"), ("gaussian", 0., 10, "random"))
LIVE_CP = np.array([0.4, 0.9, 0.12])


@pytest.fixture(scope="module")
def golden_ref():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.json")) as f:
        return json.load(f)


def test_r_known_answers_exact_gp():
    # R-package/tests/testthat/test_GPModel_gaussian_process.R:86-90, :104-107, :117-120
    coords, y = datagen.r_test_data()
    assert abs(ov.dense_neg_log_likelihood(coords, CP, y, "exponential") - 124.2549533) < 1e-6
    assert abs(ov.dense_neg_log_likelihood(coords, CP, y, "matern", 1.5) - 141.3502172) < 1e-6
    assert abs(ov.dense_neg_log_likelihood(coords, CP, y, "matern", 2.5) - 158.1111626) < 1e-6


def test_r_known_answers_vecchia():
    # :1145-1149 Vecchia m=30, ordering "none"; :1105-1111 Vecchia with m = n-1 equals the exact GP
    coords, y = datagen.r_test_data()
    o = ov.VecchiaOracle(coords, 30, "exponential", vecchia_ordering="none")
    assert abs(o.neg_log_likelihood(CP, y) - 124.2252524) < 1e-6
    o = ov.VecchiaOracle(coords, 99, "exponential", vecchia_ordering="none")
    assert abs(o.neg_log_likelihood(CP, y) - 124.2549533) < 1e-6


def test_oracle_matches_golden_nll(golden):
    for spec in golden["nll"]:
        coords, y = case_data(spec)
        o = ov.VecchiaOracle(coords, spec["num_neighbors"], spec["cov_function"], spec["cov_fct_shape"],
                             vecchia_ordering=spec["vecchia_ordering"], seed=spec.get("seed_model", spec["seed"]))
        v = o.neg_log_likelihood(np.array(spec["cov_pars"]), y)
        assert abs(v - spec["negll"]) <= 1e-10 * abs(spec["negll"]), spec


def test_oracle_gradient_is_derivative_of_nll():
    coords, y = datagen.synth(600, 2, 11)
    o = ov.VecchiaOracle(coords, 12, "matern", 1.5, vecchia_ordering="random", seed=2)
    x = np.log(np.array([1.3, 6.0]))
    f0, g, _ = o.nll_and_grad_profiled(x, y)
    for k in range(2):
        h = 1e-6
        xp, xm = x.copy(), x.copy()
        xp[k] += h; xm[k] -= h
        fd = (o.nll_and_grad_profiled(xp, y)[0] - o.nll_and_grad_profiled(xm, y)[0]) / (2 * h)
        assert abs(fd - g[k]) < 1e-5 * max(1., abs(g[k]))


def test_oracle_matches_reference_library_live(golden_ref):
    coords, y = datagen.synth(1200, 2, 21)
    recs = golden_ref["vecchia_nll"]
    assert [(r["cov_function"], r["cov_fct_shape"], r["num_neighbors"], r["vecchia_ordering"]) for r in recs] == list(LIVE_CASES)
    for r in recs:
        o = ov.VecchiaOracle(coords, r["num_neighbors"], r["cov_function"], r["cov_fct_shape"], vecchia_ordering=r["vecchia_ordering"], seed=4)
        a, b = r["negll"], o.neg_log_likelihood(LIVE_CP, y)
        assert abs(a - b) <= 1e-10 * abs(a)


def test_oracle_neighbours_sorted_and_causal():
    coords = datagen.lattice(25)
    perm = ov.random_order(coords.shape[0], 3)
    co = coords[perm]
    nn = ov.knn(co, 9)
    for i in range(co.shape[0]):
        q = min(i, 9)
        row = nn[i]
        assert (row[:q] >= 0).all() and (row[:q] < i).all() and (row[q:] == -1).all()
        if i > 9:
            d = ((co[row[:q]] - co[i]) ** 2).sum(1)
            assert (np.diff(d) >= 0).all()
