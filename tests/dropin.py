"""Staging of the UNMODIFIED reference Python package next to a chosen shared library (shared by the drop-in tests).
The package is taken from python-package/gpboost of the reference checkout oracle/_ref is built from (oracle.build.REFERENCE_DIR);
nothing of it is part of this repository."""
import json
import os
import subprocess
import sys
import tempfile
import textwrap

from oracle.build import REFERENCE_DIR


def ref_package_dir():
    pkg = os.path.join(REFERENCE_DIR, "python-package", "gpboost")
    return pkg if os.path.isdir(pkg) else None


def stage(lib_path):
    """scratch dir with gpboost/ = the reference's module files + lib_gpboost.so -> lib_path (libpath.py:36 finds it there)"""
    src = ref_package_dir()
    tmp = tempfile.mkdtemp()
    pkg = os.path.join(tmp, "gpboost")
    os.makedirs(pkg)
    for f in os.listdir(src):
        if f.endswith(".py") or f == "VERSION.txt":
            os.symlink(os.path.join(src, f), os.path.join(pkg, f))
    os.symlink(lib_path, os.path.join(pkg, "lib_gpboost.so"))
    return tmp


def run_with(lib_path, body, timeout=900):
    """runs `body` (python source that fills a dict `out`) with `import gpboost as gpb` bound to lib_path; returns out"""
    tmp = stage(lib_path)
    code = textwrap.dedent("""
        import json, os, sys, types
        sys.modules.setdefault("optuna", types.ModuleType("optuna"))   # hard import of the package, not installed here
        sys.path.insert(0, %r)
        import numpy as np
        import gpboost as gpb
        assert gpb.basic._LIB._name.endswith("lib_gpboost.so")
        out = {}
        """ % tmp) + textwrap.dedent(body) + "\nprint('RESULT' + json.dumps(out))\n"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [ln for ln in r.stdout.split("\n") if ln.startswith("RESULT")][-1]
    return json.loads(line[len("RESULT"):])
