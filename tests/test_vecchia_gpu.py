"""GPU parity tests (run with -m gpu on the B200 box). Everything goes through the C ABI of
lib_gpboost_b200.so; the oracle (and the stored results of the unmodified reference library) is only the checker.

Tolerances: neighbour indices bit-exact; negative log-likelihood <= 1e-8 relative (north_star), in practice
~1e-13; B, D^-1, gradients and Psi^-1 y <= 1e-8 relative."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import datagen
from conftest import case_data
from oracle import vecchia as ov

pytestmark = pytest.mark.gpu

REL = 1e-8
LIVE_KW = dict(cov_function="matern", cov_fct_shape=2.5, gp_approx="vecchia", num_neighbors=11, seed=6)
LIVE_CP = np.array([0.2, 1.1, 0.3])


def P(a, t=C.c_double):
    return a.ctypes.data_as(C.POINTER(t))


@pytest.fixture(scope="module")
def lib(product_lib):
    assert product_lib.gpbdev_device_count() > 0, "no CUDA device visible — GPU tests need the B200 box"
    return product_lib


@pytest.fixture(scope="module")
def golden_ref():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.json")) as f:
        return json.load(f)


def chk(lib, rc):
    assert rc == 0, lib.gpbdev_last_error().decode()


def make_engine(lib, coords, m, ordering="random", seed=1):
    n, d = coords.shape
    perm = ov.random_order(n, seed) if ordering == "random" else np.arange(n, dtype=np.int32)
    co = np.ascontiguousarray(coords[perm])
    h = C.c_void_p()
    chk(lib, lib.gpbdev_vecchia_create(C.byref(h), 0, C.c_int64(n), d, m, P(co), P(perm, C.c_int32), None, C.c_int64(0), C.c_int64(n)))
    return h, perm, co


# ---------------------------------------------------------------------------------------- neighbours
@pytest.mark.parametrize("n,d,m", [(300, 2, 10), (5000, 2, 30), (20000, 2, 20), (6000, 3, 15), (4000, 1, 8), (1200, 5, 12), (40, 2, 30),
                                   (9000, 2, 60), (5000, 3, 45), (50, 2, 60)])
def test_neighbours_bit_exact_random_coords(lib, n, d, m):
    coords, _ = datagen.synth(n, d, 9)
    m = min(m, n - 1, 60)
    h, perm, co = make_engine(lib, coords, m)
    nn = np.empty((n, m), dtype=np.int32)
    chk(lib, lib.gpbdev_vecchia_get_nn(h, P(nn, C.c_int32)))
    assert np.array_equal(nn, ov.knn(co, m))
    lib.gpbdev_vecchia_free(h)


@pytest.mark.parametrize("k,m,ordering", [(30, 12, "random"), (40, 8, "none"), (25, 30, "random"), (30, 48, "random")])
def test_neighbours_bit_exact_on_lattice_with_distance_ties(lib, k, m, ordering):
    coords = datagen.lattice(k)
    h, perm, co = make_engine(lib, coords, m, ordering, seed=2)
    nn = np.empty((coords.shape[0], m), dtype=np.int32)
    chk(lib, lib.gpbdev_vecchia_get_nn(h, P(nn, C.c_int32)))
    assert np.array_equal(nn, ov.knn(co, m))
    lib.gpbdev_vecchia_free(h)


def test_neighbours_duplicates_and_clusters(lib):
    rng = np.random.default_rng(5)
    base = rng.random((500, 2))
    coords = np.concatenate([base, base[:200], base[:50] + 1e-13, rng.random((300, 2)) * 1e-3])
    h, perm, co = make_engine(lib, coords, 10, "random", seed=3)
    nn = np.empty((coords.shape[0], 10), dtype=np.int32)
    chk(lib, lib.gpbdev_vecchia_get_nn(h, P(nn, C.c_int32)))
    assert np.array_equal(nn, ov.knn(co, 10))
    lib.gpbdev_vecchia_free(h)


# ---------------------------------------------------------------------------------------- factor / sums
@pytest.mark.parametrize("cov,shape", [("exponential", 0.5), ("matern", 1.5), ("matern", 2.5), ("gaussian", 0.)])
@pytest.mark.parametrize("n,d,m", [(700, 2, 30), (3000, 2, 17), (2500, 3, 9), (35, 2, 30), (1500, 2, 60), (900, 3, 40), (45, 2, 60)])
def test_factor_sums_and_gradient_match_oracle(lib, cov, shape, n, d, m):
    coords, y = datagen.synth(n, d, 13)
    m = min(m, n - 1)
    h, perm, co = make_engine(lib, coords, m)
    cid = ov.cov_id(cov, shape)
    s2, pt = ov.transform_cov_pars([0.4, 1.3, 0.15], cov, shape)
    chk(lib, lib.gpbdev_vecchia_set_y(h, P(np.ascontiguousarray(y))))
    nn = ov.knn(co, m)
    A, Dinv, Ag, Dg, bad = ov.factor(co, nn, cid, pt, calc_grad=True)
    assert bad == 0
    yo = y[perm]
    ref = ov.nll_from_factor(nn, A, Dinv, yo, s2)
    out = np.zeros(9)
    for mode in (0, 1, 2):
        chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), mode, P(out)))
        assert abs(out[0] - ref[1]) <= REL * abs(ref[1])
        assert abs(out[1] - ref[2]) <= REL * max(1., abs(ref[2]))
        assert out[2] == 0
    g_ref = ov.grad_from_factor(nn, A, Dinv, Ag, Dg, yo, s2)
    g = np.array([(out[3 + k] - 0.5 * out[5 + k]) / s2 + 0.5 * out[7 + k] for k in range(2)])
    assert np.all(np.abs(g - g_ref) <= REL * np.maximum(1., np.abs(g_ref)))
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 1, P(out)))
    A_d = np.empty((n, m)); Di_d = np.empty(n)
    chk(lib, lib.gpbdev_vecchia_get_factor(h, P(A_d), P(Di_d)))
    assert np.abs(A_d - A).max() <= REL
    assert (np.abs(Di_d - Dinv) / Dinv).max() <= REL
    ya = np.empty(n)
    chk(lib, lib.gpbdev_vecchia_yaux(h, P(ya)))
    ya_o = np.empty(n); ya_o[perm] = ov.yaux(nn, A, Dinv, yo)
    assert np.abs(ya - ya_o).max() <= REL * np.abs(ya_o).max()
    lib.gpbdev_vecchia_free(h)


# ---------------------------------------------------------------------------------------- C API: likelihood
def test_capi_neg_log_likelihood_golden(lib, golden):
    from gpboost_b200 import GPModel
    for spec in golden["nll"]:
        coords, y = case_data(spec)
        mdl = GPModel(gp_coords=coords, cov_function=spec["cov_function"], cov_fct_shape=spec["cov_fct_shape"], gp_approx="vecchia",
                      num_neighbors=spec["num_neighbors"], vecchia_ordering=spec["vecchia_ordering"],
                      seed=spec.get("seed_model", spec["seed"]))
        v = mdl.neg_log_likelihood(np.array(spec["cov_pars"]), y)
        assert abs(v - spec["negll"]) <= REL * abs(spec["negll"]), (spec, v)


def test_capi_r_known_answers(lib):
    # R-package/tests/testthat/test_GPModel_gaussian_process.R:1145-1149 and :1105-1111 (m = 30 of n = 100 only here)
    from gpboost_b200 import GPModel
    coords, y = datagen.r_test_data()
    mdl = GPModel(gp_coords=coords, cov_function="exponential", gp_approx="vecchia", num_neighbors=30, vecchia_ordering="none")
    assert abs(mdl.neg_log_likelihood(np.array([0.1, 1.6, 0.2]), y) - 124.2252524) < 1e-6


def test_capi_fixed_effects_and_current_negll(lib):
    from gpboost_b200 import GPModel
    coords, y = datagen.synth(1500, 2, 17)
    fe = np.sin(coords[:, 0])
    mdl = GPModel(gp_coords=coords, gp_approx="vecchia", num_neighbors=12, seed=3)
    cp = np.array([0.3, 0.8, 0.2])
    a = mdl.neg_log_likelihood(cp, y, fixed_effects=fe)
    b = mdl.neg_log_likelihood(cp, y - fe)
    assert abs(a - b) <= 1e-12 * abs(a)
    # the "current" value belongs to the optimiser: a likelihood evaluation elsewhere does not move it (as in the reference)
    mdl.fit(y)
    opt = mdl.get_current_neg_log_likelihood()
    assert opt < b
    mdl.neg_log_likelihood(cp, y)
    assert mdl.get_current_neg_log_likelihood() == opt


# ---------------------------------------------------------------------------------------- C API: fit
def test_capi_fit_matches_reference_golden(lib, golden):
    """Same optimum as the reference's L-BFGS run: NLL to 1e-6 relative, parameters to 1e-3 relative.
    (The iteration path is decision-dependent; the iteration count is reported, and asserted within +-3.)"""
    from gpboost_b200 import GPModel
    for spec in golden["fit"]:
        coords, y = case_data(spec)
        mdl = GPModel(gp_coords=coords, cov_function=spec["cov_function"], cov_fct_shape=spec["cov_fct_shape"], gp_approx="vecchia",
                      num_neighbors=spec["num_neighbors"], vecchia_ordering=spec["vecchia_ordering"],
                      seed=spec.get("seed_model", spec["seed"]))
        mdl.fit(y)
        cp = mdl.get_cov_pars()
        nll = mdl.get_current_neg_log_likelihood()
        print(spec["data"], spec["cov_function"], "iters", mdl._get_num_optim_iter(), "ref", spec["num_it"], cp, spec["cov_pars"])
        assert abs(nll - spec["negll"]) <= 1e-6 * abs(spec["negll"]), (spec, nll)
        assert np.all(np.abs(cp - np.array(spec["cov_pars"])) <= 2e-3 * np.abs(spec["cov_pars"])), (spec, cp)
        assert abs(mdl._get_num_optim_iter() - spec["num_it"]) <= 3
        # the reported optimum is consistent with a fresh evaluation at the returned parameters
        assert abs(mdl.neg_log_likelihood(cp, y) - nll) <= 1e-9 * abs(nll)


def test_capi_response_gradient_matches_oracle(lib):
    from gpboost_b200 import GPModel
    coords, y = datagen.synth(2500, 2, 23)
    mdl = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=14, seed=5)
    cp0 = np.array([0.35, 0.9, 0.18])
    mdl.set_optim_params({"init_cov_pars": cp0, "maxit": 0})
    mdl.fit(y)  # maxit = 0: parameters stay at init_cov_pars
    g = mdl.response_gradient(y)
    o = ov.VecchiaOracle(coords, 14, "matern", 1.5, "random", 5)
    ya, s2 = o.grad_response(cp0, y)
    assert np.abs(g - ya / s2).max() <= REL * np.abs(ya / s2).max()


def test_capi_live_against_reference_library(lib, golden_ref):
    from gpboost_b200 import GPModel
    coords, y = datagen.synth(2500, 2, 29)
    a = GPModel(gp_coords=coords, **LIVE_KW)
    rec = golden_ref["vecchia_capi"]
    va, vb = a.neg_log_likelihood(LIVE_CP, y), rec["negll"]
    assert abs(va - vb) <= REL * abs(vb)
    a.fit(y)
    assert abs(a.get_current_neg_log_likelihood() - rec["fit_negll"]) <= 1e-6 * abs(rec["fit_negll"])


# ---------------------------------------------------------------------------------------- edge cases
def test_edge_cases(lib):
    from gpboost_b200 import GPModel, GPBoostError
    coords, y = datagen.synth(12, 2, 31)
    mdl = GPModel(gp_coords=coords, gp_approx="vecchia", num_neighbors=30, vecchia_ordering="none")  # m clipped to n-1
    o = ov.VecchiaOracle(coords, 11, "matern", 1.5, "none")
    cp = np.array([0.5, 1., 0.3])
    assert abs(mdl.neg_log_likelihood(cp, y) - o.neg_log_likelihood(cp, y)) <= REL * 50
    with pytest.raises(GPBoostError):
        GPModel(gp_coords=datagen.synth(100, 2, 1)[0], gp_approx="vecchia", num_neighbors=61)  # engine limit: 60
    with pytest.raises(GPBoostError):
        mdl.neg_log_likelihood(np.array([0.5, -1., 0.3]), y)
    with pytest.raises(ValueError):
        mdl.neg_log_likelihood(cp, y[:5])


# ---------------------------------------------------------------------------------------- full size (BASELINE config 2)
def test_full_size_properties_n1e6(lib):
    """n = 1e6, m = 30, Matern-1.5 (BASELINE.json configs[1]): the oracle is too slow to factor this in a test, so
    size-independent properties are checked: neighbour causality/sortedness, quad-form homogeneity,
    linearity of Psi^-1, and y^T(Psi^-1 y) = quad form."""
    n, m = 1000000, 30
    rng = np.random.default_rng(1)
    coords = rng.random((n, 2)); y = rng.standard_normal(n)
    h, perm, co = make_engine(lib, coords, m)
    nn = np.empty((n, m), dtype=np.int32)
    chk(lib, lib.gpbdev_vecchia_get_nn(h, P(nn, C.c_int32)))
    rows = np.arange(n)[:, None]
    assert (nn[m + 1:] >= 0).all() and (nn[m + 1:] < rows[m + 1:]).all()
    idx = rng.integers(m + 1, n, 2000)
    d2 = ((co[nn[idx]] - co[idx][:, None, :]) ** 2).sum(-1)
    assert (np.diff(d2, axis=1) >= 0).all()
    # sampled rows agree with an independent brute-force search
    for i in idx[:40]:
        dd = ((co[:i] - co[i]) ** 2).sum(1)
        assert set(np.argsort(dd, kind="stable")[:m]) == set(nn[i])
    cid = ov.cov_id("matern", 1.5)
    s2, pt = ov.transform_cov_pars([0.5, 1.0, 0.1], "matern", 1.5)
    out1, out2 = np.zeros(9), np.zeros(9)
    chk(lib, lib.gpbdev_vecchia_set_y(h, P(y)))
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 1, P(out1)))
    ya = np.empty(n); chk(lib, lib.gpbdev_vecchia_yaux(h, P(ya)))
    assert abs(y @ ya - out1[0]) <= 1e-10 * out1[0]
    y2 = rng.standard_normal(n)
    chk(lib, lib.gpbdev_vecchia_set_y(h, P(3. * y)))
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 0, P(out2)))
    assert abs(out2[0] - 9. * out1[0]) <= 1e-12 * out2[0] and out2[1] == out1[1]
    chk(lib, lib.gpbdev_vecchia_set_y(h, P(2. * y - 0.5 * y2)))
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 1, P(out2)))
    yb = np.empty(n); chk(lib, lib.gpbdev_vecchia_yaux(h, P(yb)))
    chk(lib, lib.gpbdev_vecchia_set_y(h, P(y2)))
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 1, P(out2)))
    yc = np.empty(n); chk(lib, lib.gpbdev_vecchia_yaux(h, P(yc)))
    assert np.abs(yb - (2. * ya - 0.5 * yc)).max() <= 1e-10 * np.abs(ya).max()
    # modes agree with each other on the shared sums
    chk(lib, lib.gpbdev_vecchia_eval(h, cid, C.c_double(pt[0]), C.c_double(pt[1]), 2, P(out1)))
    # (the passes run on different grids — resident CTAs per SM differ — so the fixed summation order differs between modes)
    assert abs(out1[0] - out2[0]) <= 1e-13 * out2[0] and abs(out1[1] - out2[1]) <= 1e-13 * abs(out2[1])
    lib.gpbdev_vecchia_free(h)


def test_full_size_against_golden_subsample_consistency(lib):
    """n = 2e5 through the C API against the oracle (the largest size the C oracle factors in a few seconds)."""
    from gpboost_b200 import GPModel
    coords, y = datagen.synth(200000, 2, 37)
    mdl = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=30, seed=1)
    cp = np.array([0.5, 1.0, 0.1])
    got = mdl.neg_log_likelihood(cp, y)
    want = ov.VecchiaOracle(coords, 30, "matern", 1.5, "random", 1).neg_log_likelihood(cp, y)
    assert abs(got - want) <= REL * abs(want)
