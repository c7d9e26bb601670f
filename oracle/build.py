"""TEST INFRASTRUCTURE ONLY — builds the oracle's C restatement (liborc.so) and, where /root/reference
exists (the build container, not the GPU box), the unmodified reference library (oracle/_ref/lib_gpboost.so)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)
_SRCS = ["vecchia_oracle.c", "tree_oracle.c"]
_CXX_SRCS = ["shuffle_oracle.cpp"]
# checkout of the unmodified reference: oracle/_ref is built from its sources and the drop-in tests take its Python package;
# GPBOOST_REFERENCE names a checkout elsewhere
REFERENCE_DIR = os.environ.get("GPBOOST_REFERENCE", "/root/reference")


def oracle_lib_path():
    return os.path.join(_HERE, "liborc.so")


def ref_lib_path():
    return os.path.join(_HERE, "_ref", "lib_gpboost.so")


def build_oracle(force=False):
    """gcc -O2 -fopenmp the C restatement into oracle/liborc.so (seconds)."""
    out = oracle_lib_path()
    srcs = [os.path.join(_HERE, s) for s in _SRCS if os.path.exists(os.path.join(_HERE, s))]
    deps = srcs + [os.path.join(_HERE, s) for s in _CXX_SRCS]
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in deps):
        return out
    # -ffp-contract=off: keep mul/add unfused like the reference's x86-64 baseline build
    objs = []
    for s in srcs:
        o = s[:-2] + ".o"
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-fopenmp", "-fPIC", "-ffp-contract=off", "-c", s, "-o", o])
        objs.append(o)
    for s in _CXX_SRCS:
        s = os.path.join(_HERE, s)
        o = s[:-4] + ".o"
        subprocess.check_call(["/usr/bin/g++", "-O2", "-fPIC", "-c", s, "-o", o])
        objs.append(o)
    subprocess.check_call(["/usr/bin/g++", "-shared", "-fopenmp", "-o", out] + objs + ["-lm"])
    return out


def build_ref(jobs=8):
    """Build the unmodified reference into oracle/_ref/ (≈6 min). No-op when already built or when
    /root/reference is absent (GPU box: the prebuilt .so travels with the snapshot)."""
    out = ref_lib_path()
    if os.path.exists(out):
        return out
    if not os.path.isdir(os.path.join(REFERENCE_DIR, "src")):
        return None
    subprocess.check_call(["make", "-f", os.path.join(_HERE, "Makefile.ref"), "-j%d" % jobs,
                           "REF=" + REFERENCE_DIR, "OUT=" + os.path.join(_HERE, "_ref")], cwd=_REPO,
                          stdout=subprocess.DEVNULL)
    return out
