"""Drop-in boundary, exercised with the UNMODIFIED reference Python package (python-package/gpboost of the reference checkout
oracle/_ref is built from, imported in place — nothing is copied): its module files are symlinked into a scratch directory next to
lib_gpboost_b200.so under the name the package searches for (lib_gpboost.so, libpath.py:36). The package must import (every symbol it
binds at load time resolves), build a Dataset through LGBM_DatasetCreateFromMat / SetField / GetField on the host, and reach the device-creating entries —
which, on this GPU-less container, must fail through the reference's own error channel (GPBoostError from LGBM_GetLastError)
because the library has no CPU fallback. Skipped where there is no reference checkout."""
import os
import subprocess
import sys
import tempfile
import textwrap

import pytest

import dropin

REF_PKG = dropin.ref_package_dir()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(REF_PKG is None, reason="reference Python package not present (set GPBOOST_REFERENCE)")
def test_unmodified_reference_package_loads_and_reaches_the_device_entries():
    lib = os.path.join(ROOT, "gpboost_b200", "lib_gpboost_b200.so")
    assert os.path.exists(lib)
    tmp = tempfile.mkdtemp()
    pkg = os.path.join(tmp, "gpboost")
    os.makedirs(pkg)
    for f in os.listdir(REF_PKG):
        if f.endswith(".py") or f == "VERSION.txt":
            os.symlink(os.path.join(REF_PKG, f), os.path.join(pkg, f))
    os.symlink(lib, os.path.join(pkg, "lib_gpboost.so"))
    code = textwrap.dedent("""
        import sys, types
        sys.modules.setdefault("optuna", types.ModuleType("optuna"))   # hard import of the package, not installed here
        sys.path.insert(0, %r)
        import numpy as np
        import gpboost as gpb
        assert gpb.basic._LIB._name.endswith("lib_gpboost.so")
        ds = gpb.Dataset(np.random.default_rng(1).random((100, 3)), np.arange(100) / 100.)
        ds.construct()
        assert ds.num_data() == 100 and ds.num_feature() == 3
        assert abs(float(ds.get_label()[7]) - 0.07) < 1e-6
        import torch
        has_gpu = torch.cuda.is_available()
        out = []
        for make in (lambda: gpb.GPModel(gp_coords=np.random.default_rng(0).random((200, 2)), cov_function="matern", cov_fct_shape=1.5,
                                         gp_approx="vecchia", num_neighbors=10),
                     lambda: gpb.Booster(params={"objective": "regression_l2", "num_leaves": 8, "verbose": -1}, train_set=ds)):
            try:
                make()
                out.append("created")
            except gpb.basic.GPBoostError as e:
                out.append("error: " + str(e))
        print(has_gpu, out)
        if not has_gpu:
            assert all(o.startswith("error") and "no CPU fallback" in o for o in out), out
        else:
            assert out == ["created", "created"], out
        """ % tmp)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.skipif(REF_PKG is None, reason="reference Python package not present (set GPBOOST_REFERENCE)")
def test_unmodified_reference_package_predicts_through_the_library(ref_lib):
    """gpb.Booster(model_str=...) / predict / save_model / Booster(model_file=...) of the unmodified package, bound to THIS library,
    on a model trained by the reference: predictions equal the reference library's own (host path, no device needed)."""
    if ref_lib is None:
        pytest.skip("reference library not built")
    import numpy as np
    from gpboost_b200.booster import Booster, Dataset
    rng = np.random.default_rng(0)
    X = rng.random((800, 4)); y = np.sin(3 * X[:, 0]) + X[:, 1] ** 2 + 0.1 * rng.standard_normal(800)
    params = dict(objective="regression", num_leaves=7, min_data_in_leaf=20, learning_rate=0.1, max_bin=255, verbose=-1)
    b = Booster(params, Dataset(X, y, params=params, _lib=ref_lib), _lib=ref_lib)
    for _ in range(5):
        b.update()
    Xt = np.random.default_rng(3).random((50, 4))
    want = b.predict(Xt)
    lib = os.path.join(ROOT, "gpboost_b200", "lib_gpboost_b200.so")
    tmp = tempfile.mkdtemp()
    pkg = os.path.join(tmp, "gpboost")
    os.makedirs(pkg)
    for f in os.listdir(REF_PKG):
        if f.endswith(".py") or f == "VERSION.txt":
            os.symlink(os.path.join(REF_PKG, f), os.path.join(pkg, f))
    os.symlink(lib, os.path.join(pkg, "lib_gpboost.so"))
    with open(os.path.join(tmp, "model.txt"), "w") as f:
        f.write(b.model_to_string())
    np.save(os.path.join(tmp, "Xt.npy"), Xt); np.save(os.path.join(tmp, "want.npy"), want)
    code = textwrap.dedent("""
        import os, sys, types
        sys.modules.setdefault("optuna", types.ModuleType("optuna"))
        tmp = %r
        sys.path.insert(0, tmp)
        import numpy as np
        import gpboost as gpb
        Xt = np.load(os.path.join(tmp, "Xt.npy")); want = np.load(os.path.join(tmp, "want.npy"))
        bst = gpb.Booster(model_str=open(os.path.join(tmp, "model.txt")).read())
        assert bst.num_trees() == 5 and bst.num_feature() == 4 and bst.feature_name() == ["Column_%%d" %% i for i in range(4)]
        assert np.array_equal(bst.predict(Xt), want)
        bst.save_model(os.path.join(tmp, "m2.txt"))
        assert np.array_equal(gpb.Booster(model_file=os.path.join(tmp, "m2.txt")).predict(Xt), want)
        """ % tmp)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
