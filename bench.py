#!/usr/bin/env python
"""bench.py — GP log-likelihood evaluations/s on BASELINE.json configs[1]:
Vecchia GP, n = 1e6, 2-D coords U[0,1]^2, m = 30 neighbours, Matern-1.5, Gaussian likelihood, random ordering.

A "step" = one pass of the hot path = one negative-log-likelihood evaluation at fixed covariance parameters
(covariance blocks + batched local Cholesky + quadratic form + log-det; SURVEY §8d metric (ii)).

  value : device-resident throughput — y already in HBM, K passes timed with CUDA events on the engine's stream,
          L2 flushed (256 MiB write) before every timed pass.
  e2e   : the same metric through the reference-facing C API call GPB_EvalNegLogLikelihood with a pinned HOST
          response vector: H2D of y (8 MB) + pass + D2H of the sums inside the timed region, every step.
  N > 1 : one process per GPU (torchrun); the ordered observations are row-sharded, each rank evaluates its rows and
          the 9 fp64 sums are all-reduced over NCCL (strong scaling at fixed n = 1e6).
  --impl reference : the UNMODIFIED reference CPU library (oracle/_ref/lib_gpboost.so) on the host cores, same call.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_OBS = 1000000
M_NEIGH = 30
COV_PARS = np.array([0.5, 1.0, 0.1])  # (sigma^2, sigma_1^2, rho): SURVEY §8d C2
WORKLOAD = "configs[1]: Vecchia GP n=1e6, d=2, m=30, Matern-1.5, Gaussian likelihood, random ordering (seed 1)"
# algorithmic work per observation, SURVEY §8(d): B not materialised (fused NLL): 4m + 8d + 8 = 144 B; ~24 kflop
ALGO_BYTES_PER_OBS = 4 * M_NEIGH + 8 * 2 + 8
ALGO_FLOPS_PER_OBS = 24e3


def host_cores():
    """Usable host cores: CPU affinity capped by the cgroup CPU quota (the GPU boxes expose 128 CPUs under a 16-CPU quota;
    running the reference's OpenMP loops with 128 threads there is several hundred times slower than with 16)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def make_data(n):
    rng = np.random.default_rng(1)
    return rng.random((n, 2)), rng.standard_normal(n)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.stop_flag = False
        self.rows = []
        self.index = index

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def time_reference(n, steps, warmup, threads):
    """The reference's own CPU implementation through the identical C API call."""
    from gpboost_b200 import GPModel
    from gpboost_b200.libpath import load_lib
    from oracle import ref_lib_path
    if not os.path.exists(ref_lib_path()):
        return None
    ref = load_lib(ref_lib_path())
    coords, y = make_data(n)
    t0 = time.perf_counter()
    mdl = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=M_NEIGH,
                  vecchia_ordering="random", seed=1, num_parallel_threads=threads, _lib=ref)
    t_create = time.perf_counter() - t0
    for _ in range(warmup):
        mdl.neg_log_likelihood(COV_PARS, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        v = mdl.neg_log_likelihood(COV_PARS, y)
    dt = (time.perf_counter() - t0) / steps
    return {"sec_per_eval": dt, "negll": v, "create_s": t_create}


def time_dense(n, lib, threads, reps=5):
    """BASELINE configs[0]: exact GP (gp_approx="none"), n = 2000, 2-D Matern-1.5: one GPB_EvalNegLogLikelihood = Gram build +
    dense Cholesky + solves; and one GPB_OptimCovPar (fit)."""
    from gpboost_b200 import GPModel
    rng = np.random.default_rng(1)
    coords = rng.random((n, 2))
    y = np.sin(5 * coords[:, 0]) * np.cos(4 * coords[:, 1]) + 0.5 * rng.standard_normal(n)
    mdl = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="none", num_parallel_threads=threads, _lib=lib)
    cp = np.array([0.25, 1.0, 0.1])
    v = mdl.neg_log_likelihood(cp, y)
    t0 = time.perf_counter()
    for _ in range(reps):
        v = mdl.neg_log_likelihood(cp, y)
    dt = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    mdl.fit(y)
    t_fit = time.perf_counter() - t0
    res = {"sec_per_eval": dt, "negll": v, "fit_s": t_fit, "fit_iters": mdl._get_num_optim_iter(), "fit_cov_pars": mdl.get_cov_pars().tolist()}
    if lib is None:
        flops = n ** 3 / 3.0 + 30.0 * n * n  # Cholesky n^3/3 + Gram build (~30 flop per entry incl. exp)
        res["roofline"] = {"bound": "fp64_tensor", "achieved": flops / dt / 1e12, "unit": "TFLOP/s", "flops": flops,
                           "note": "whole GPB_EvalNegLogLikelihood call (Gram + blocked Cholesky with DMMA trailing updates + solves), wall clock; at "
                                   "n = 2000 the 32 panel steps are launch-latency bound, not tensor bound"}
    return res


def time_gpboost(n, iters, lib, threads, F=50, f32=False):
    """One GPBoost iteration = LGBM_BoosterUpdateOneIter with a Vecchia GP (m=30) attached: covariance re-fit (L-BFGS) +
    Psi^-1(F - y) + one 31-leaf tree on n x 50 features (BASELINE configs[3] shape on one GPU, metric (i) of SURVEY §8d)."""
    from gpboost_b200 import GPModel
    from gpboost_b200.booster import Booster, Dataset
    rng = np.random.default_rng(1)
    coords = rng.random((n, 2))
    X = rng.random((n, F), dtype=np.float32) if f32 else rng.random((n, F))  # float32 features halve the host memory of configs[3]
    y = 2 * np.sin(3 * X[:, 0]) + X[:, 1].astype(np.float64) ** 2 + np.sin(5 * coords[:, 0]) * np.cos(4 * coords[:, 1]) + 0.5 * rng.standard_normal(n)
    params = dict(objective="regression", num_leaves=31, min_data_in_leaf=20, learning_rate=0.1, max_bin=255, verbose=-1)
    if lib is not None:
        params["num_threads"] = threads
    gp = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=M_NEIGH,
                 vecchia_ordering="random", seed=1, num_parallel_threads=threads, _lib=lib)
    b = Booster(params, Dataset(X, y, params=params, _lib=lib), gp_model=gp, _lib=lib)
    t0 = time.perf_counter(); b.update(); first = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(iters):
        b.update()
    dt = (time.perf_counter() - t0) / iters
    out = {"sec_per_iter": dt, "first_iter_s": first, "cov_pars": gp.get_cov_pars().tolist()}
    if lib is None:
        out["hist_roofline"] = hist_roofline(b)
    return out


def hist_roofline(booster):
    """Roofline of the tree side's dominant kernel: the root-pass histogram kernel timed alone with CUDA events (L2 flushed before every
    launch). Algorithmic bytes per row (SURVEY §8d): the row's bins (Fpad) + its gradient (8)."""
    ms, row_bytes, rows = C.c_float(0), C.c_int(0), C.c_int64(0)
    L = booster._LIB
    if L.GPB200_BoosterTimeRootHistogram(booster.handle, 10, C.byref(ms), C.byref(row_bytes), C.byref(rows)) != 0:
        return {"error": L.LGBM_GetLastError().decode()}
    hbm_peak, src = measured_hbm_peak()
    ach = rows.value * row_bytes.value / (ms.value * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "hist3_kernel (root pass, all rows of this rank)", "kernel_ms": ms.value,
            "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": None,
            "algorithmic_bytes_per_row": row_bytes.value, "rows": rows.value, "peak_source": src,
            "note": "shared-memory (LSU) bound: one read-modify-write per (row, feature) on private fp64 histograms"}


def measured_hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s"


def time_gpboost_grouped(n, iters, lib, threads, F=50, groups=10000):
    """BASELINE configs[2]: GPBoost with a single-level grouped random effect (1e4 groups), n x 50 features, 31-leaf trees;
    one iteration = LGBM_BoosterUpdateOneIter (variance re-fit + Psi^-1(F - y) + one tree). Also times the same data without
    a random-effects model (tree side alone)."""
    from gpboost_b200 import GPModel
    from gpboost_b200.booster import Booster, Dataset
    rng = np.random.default_rng(1)
    X = rng.random((n, F))
    group = rng.integers(0, groups, size=n)
    y = 2 * np.sin(3 * X[:, 0]) + X[:, 1] ** 2 + rng.standard_normal(groups)[group] + 0.5 * rng.standard_normal(n)
    params = dict(objective="regression", num_leaves=31, min_data_in_leaf=20, learning_rate=0.1, max_bin=255, verbose=-1)
    if lib is not None:
        params["num_threads"] = threads
    ds = Dataset(X, y, params=params, _lib=lib)
    out = {}
    for key, gp in (("grouped", GPModel(group_data=group, num_parallel_threads=threads, _lib=lib)), ("trees_only", None)):
        b = Booster(params, ds, gp_model=gp, _lib=lib)
        t0 = time.perf_counter(); b.update(); first = time.perf_counter() - t0
        t0 = time.perf_counter()
        for _ in range(iters):
            b.update()
        out[key] = {"sec_per_iter": (time.perf_counter() - t0) / iters, "first_iter_s": first}
        if gp is not None:
            out[key]["cov_pars"] = gp.get_cov_pars().tolist()
        elif lib is None:
            out[key]["hist_roofline"] = hist_roofline(b)
        del b
    return out


def time_laplace(n, lib, threads, reps=1, barrier=None):
    """BASELINE configs[4]: bernoulli_logit likelihood + latent Vecchia GP (m=30), one Laplace-approximated likelihood
    evaluation = Newton mode finding (VADU-PCG) + log-determinant by stochastic Lanczos quadrature (50 probes), through
    GPB_EvalNegLogLikelihood with host buffers. Same call, same defaults for both libraries."""
    from gpboost_b200 import GPModel
    rng = np.random.default_rng(5)
    coords = rng.random((n, 2))
    latent = 1.5 * np.sin(6 * coords[:, 0]) * np.cos(4 * coords[:, 1]) + 0.3 * rng.standard_normal(n)
    y = (rng.random(n) < 1. / (1. + np.exp(-latent))).astype(np.float64)
    t0 = time.perf_counter()
    gp = GPModel(likelihood="bernoulli_logit", gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia",
                 num_neighbors=M_NEIGH, vecchia_ordering="random", seed=1, matrix_inversion_method="iterative",
                 num_parallel_threads=threads, _lib=lib)
    t_create = time.perf_counter() - t0
    pars = np.array([1.0, 0.05])
    t0 = time.perf_counter(); v = gp.neg_log_likelihood(pars, y); first = time.perf_counter() - t0
    if barrier:
        barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        v = gp.neg_log_likelihood(pars, y)
    if barrier:
        barrier()
    dt = (time.perf_counter() - t0) / reps
    out = {"n": n, "sec_per_eval": dt, "first_eval_s": first, "create_s": t_create, "negll": v}
    if lib is None:
        info = gp.laplace_info()
        out.update({"newton_it": int(info[1]), "cg_it": int(info[2]), "slq_it": int(info[3])})
        # roofline of the dominant kernels: one operator and one preconditioner application on the probe block, CUDA events.
        # Compulsory bytes per row (SURVEY §8d): two passes over B (coefficients 8 B + indices 4 B per entry, m+1 entries) + four
        # t-column vector rows read or written.
        L = gp._LIB
        eng = gp.device_engine()
        t_cols = 50 // max(1, int(os.environ.get("WORLD_SIZE", "1")))
        hbm_peak, src = measured_hbm_peak()
        roof = {}
        for label, tc in (("probe_block", None), ("newton_vector", 1)):
            ms = (C.c_float * 2)()
            tcols = tc if tc is not None else -1
            # the probe count of this rank is whatever set_probes received; ask with t = 1 first, then the block size
            rc = -1
            for cand in ([1] if tc == 1 else [t_cols, t_cols + 1, 50]):
                rc = L.gpbdev_vecchia_laplace_time_ops(eng, cand, 5, ms)
                if rc == 0:
                    tcols = cand
                    break
            if rc != 0:
                continue
            algo = n * (2 * 12 * (M_NEIGH + 1) + 4 * 8 * tcols)
            for k, nm in ((0, "operator"), (1, "preconditioner")):
                ach = algo / (ms[k] * 1e-3) / 1e9
                roof["%s_%s" % (label, nm)] = {"bound": "hbm", "kernel_ms": ms[k], "t": tcols, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                                               "frac": ach / hbm_peak, "algorithmic_bytes": algo, "peak_source": src}
        roof["note"] = ("operator = mv_B + mv_Bt kernels, preconditioner = the two sparse triangular solves; every row gathers m neighbour rows, "
                        "so DRAM/L2 traffic is up to (m+1)/2 times the compulsory bytes when the block does not fit L2; t = 1 is latency bound")
        out["roofline"] = roof
    return out


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the likelihood kernel (n=1e6, one launch) from the committed
    `ncu --set full` capture summary (profiles/r02_ncu_raw_summary.txt, section prof_nll2); None when the file is not there."""
    try:
        tot, inside = 0.0, False
        for ln in open(os.path.join(ROOT, "profiles", "r02_ncu_raw_summary.txt")):
            if ln.startswith("=="):
                inside = "prof_nll2" in ln
            elif inside and ("dram__bytes_read.sum" in ln or "dram__bytes_write.sum" in ln):
                val, unit = ln.split("=")[1].split()[:2]
                tot += float(val) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
        return tot if tot > 0 else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample-n", type=int, default=250000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--boost-n", type=int, default=1000000, help="n of the GPBoost-iteration measurement (0 = skip)")
    ap.add_argument("--boost-features", type=int, default=50, help="features of the GPBoost-iteration measurements (BASELINE configs[3]: --boost-n 5000000 --boost-features 100 on 8 GPUs)")
    ap.add_argument("--boost-ref-n", type=int, default=100000, help="--impl reference: n of the GPBoost-Vecchia iteration sub-problem (0 = skip)")
    ap.add_argument("--grouped-ref-n", type=int, default=1000000, help="--impl reference: n of the grouped-RE GPBoost iterations (configs[2] is cheap on the CPU: full size; 0 = skip)")
    ap.add_argument("--config3", default="auto", choices=["auto", "on", "off"], help="BASELINE configs[3] (n=5e6 x 100 features, Vecchia m=30 + trees): auto = when launched on 8 GPUs")
    ap.add_argument("--dense-n", type=int, default=2000, help="n of the exact-GP measurement (BASELINE configs[0]; 0 = skip; --impl reference times it too)")
    ap.add_argument("--laplace-n", type=int, default=1000000, help="n of the Laplace-Vecchia (bernoulli_logit) measurement, BASELINE configs[4] (0 = skip)")
    ap.add_argument("--laplace-ref-n", type=int, default=100000, help="--impl reference: n of the Laplace-Vecchia evaluation sub-problem (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed in their last step to DIR/<name>.npy (float64), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = host_cores()
    os.environ.setdefault("OMP_NUM_THREADS", str(ncores))  # before the reference library (libgomp) is loaded
    W = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        res = time_reference(N_OBS, args.steps, max(args.warmup, 1), ncores)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/lib_gpboost.so missing (build it with oracle/Makefile.ref)"}))
            return 0
        v = 1.0 / res["sec_per_eval"]
        line = ({
            "impl": "reference", "metric": "gp_loglik_evals_per_sec", "value": v, "unit": "evals/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": res["sec_per_eval"] * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "host_threads": ncores, "model_creation_s": res["create_s"]},
            "cpu_baseline": {"value": v, "unit": "evals/s", "cores": ncores, "kind": "reference",
                             "sample": "full workload n=1e6, %d timed GPB_EvalNegLogLikelihood calls" % args.steps},
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "negll": res["negll"]})
        # BASELINE metric (i), iterations/s of LGBM_BoosterUpdateOneIter, on stated sub-problems (bounded CPU time; per-iteration cost of
        # both configurations is linear in n, so `scaled_to_n1e6` = value * n / 1e6 is given beside the measured number)
        from gpboost_b200.libpath import load_lib
        from oracle import ref_lib_path
        if args.grouped_ref_n > 0:
            ggr = time_gpboost_grouped(args.grouped_ref_n, 5, load_lib(ref_lib_path()), ncores)
            ips = 1.0 / ggr["grouped"]["sec_per_iter"]
            line["gpboost_grouped"] = {"iters_per_sec": ips, "ms_per_iter": ggr["grouped"]["sec_per_iter"] * 1e3,
                                       "trees_only_ms_per_iter": ggr["trees_only"]["sec_per_iter"] * 1e3, "n": args.grouped_ref_n,
                                       "scaled_to_n1e6": ips * args.grouped_ref_n / 1e6, "cores": ncores,
                                       "sample": "configs[2] shape (1e4 groups, 50 features, 31 leaves) at n=%d, 5 timed iterations after the first" % args.grouped_ref_n}
        if args.boost_ref_n > 0:
            gb = time_gpboost(args.boost_ref_n, 2, load_lib(ref_lib_path()), ncores)
            ips = 1.0 / gb["sec_per_iter"]
            line["gpboost"] = {"iters_per_sec": ips, "ms_per_iter": gb["sec_per_iter"] * 1e3, "n": args.boost_ref_n, "first_iter_s": gb["first_iter_s"],
                               "scaled_to_n1e6": ips * args.boost_ref_n / 1e6, "cores": ncores,
                               "sample": "GPBoost Vecchia m=30 + 31-leaf trees on n x 50 features at n=%d (sub-problem of the n=1e6 workload), "
                                         "2 timed iterations after the first, covariance parameters re-fitted every iteration" % args.boost_ref_n}
        if args.dense_n > 0:
            from gpboost_b200.libpath import load_lib
            from oracle import ref_lib_path
            dr = time_dense(args.dense_n, load_lib(ref_lib_path()), ncores, reps=2)
            line["dense"] = {"evals_per_sec": 1.0 / dr["sec_per_eval"], "n": args.dense_n, **dr}
        if args.laplace_ref_n > 0:
            from gpboost_b200.libpath import load_lib
            from oracle import ref_lib_path
            lp = time_laplace(args.laplace_ref_n, load_lib(ref_lib_path()), ncores, reps=1)
            line["laplace"] = {"evals_per_sec": 1.0 / lp["sec_per_eval"], **lp, "cores": ncores,
                               "scaled_to_n1e6": (1.0 / lp["sec_per_eval"]) * args.laplace_ref_n / 1e6,
                               "sample": "configs[4] shape at n=%d (sub-problem), one timed GPB_EvalNegLogLikelihood after the first; the iteration "
                                         "counts grow with n, so linear scaling to 1e6 flatters the reference" % args.laplace_ref_n}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    from gpboost_b200 import GPModel, load_lib
    lib = load_lib()
    if lib.gpbdev_device_count() <= local_rank:
        raise RuntimeError("bench.py: CUDA device %d not available — the B200 path has no CPU fallback" % local_rank)
    torch.cuda.set_device(local_rank)
    cb_keep = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world)
        from gpboost_b200.parallel import init_nccl
        init_nccl(lib, dist, local_rank)  # NCCL communicator owned by the C++ runtime: device-side all-reduces, no Python in the loop
    assert lib.GPB200_SetDevice(local_rank) == 0

    coords, y = make_data(N_OBS)
    t0 = time.perf_counter()
    mdl = GPModel(gp_coords=coords, cov_function="matern", cov_fct_shape=1.5, gp_approx="vecchia", num_neighbors=M_NEIGH,
                  vecchia_ordering="random", seed=1)
    t_create = time.perf_counter() - t0
    eng = mdl.device_engine()
    # pinned host response (the e2e input buffer)
    y_pin = torch.from_numpy(y).pin_memory()
    y_ptr = C.cast(y_pin.data_ptr(), C.POINTER(C.c_double))
    cp = np.ascontiguousarray(COV_PARS)
    cp_ptr = cp.ctypes.data_as(C.POINTER(C.c_double))
    negll = C.c_double(0)

    def chk(rc):
        if rc != 0:
            raise RuntimeError((lib.gpbdev_last_error() or lib.LGBM_GetLastError()).decode())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        chk(lib.gpbdev_vecchia_sync(eng))

    # transformed parameters for the device-only timing (cov_fcts.h:485-552)
    var_t, range_t = COV_PARS[1] / COV_PARS[0], np.sqrt(3.) / COV_PARS[2]
    chk(lib.GPB_EvalNegLogLikelihood(mdl.handle, y_ptr, cp_ptr, None, C.byref(negll)))  # y resident afterwards
    negll_value = negll.value

    # ---- device-resident timing (value) + per-kernel CUDA-event duration (roofline)
    for _ in range(W):
        chk(lib.gpbdev_vecchia_eval_async(eng, 1, C.c_double(var_t), C.c_double(range_t), 0))
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    launches0 = lib.gpbdev_vecchia_launch_count(eng)
    ms = C.c_float(0)
    kernel_ms = []
    barrier()
    for _ in range(args.steps):
        chk(lib.gpbdev_vecchia_flush_l2(eng))
        chk(lib.gpbdev_vecchia_timer_start(eng))
        chk(lib.gpbdev_vecchia_eval_async(eng, 1, C.c_double(var_t), C.c_double(range_t), 0))
        chk(lib.gpbdev_vecchia_timer_stop(eng, C.byref(ms)))
        kernel_ms.append(ms.value)
    barrier()
    outputs = {}  # --dump-outputs: name -> array of the last timed step
    sums = np.zeros(9)
    chk(lib.gpbdev_vecchia_get_sums(eng, sums.ctypes.data_as(C.POINTER(C.c_double))))
    outputs["vecchia_nll_sums"] = sums[:3]  # y' Psi^-1 y, log|Psi|, #(D_i <= 0) of the last device-resident pass
    dev_ms = float(np.mean(kernel_ms))
    launches = lib.gpbdev_vecchia_launch_count(eng) - launches0  # factor + reduction kernel per step (L2-flush fills not counted)
    # ---- e2e timing through the C API with host buffers
    for _ in range(W):
        chk(lib.GPB_EvalNegLogLikelihood(mdl.handle, y_ptr, cp_ptr, None, C.byref(negll)))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        chk(lib.GPB_EvalNegLogLikelihood(mdl.handle, y_ptr, cp_ptr, None, C.byref(negll)))
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    outputs["negll_e2e"] = np.array([negll.value])
    # the same call with the response in ordinary (pageable) numpy memory — what a ctypes caller of the reference's package passes;
    # the engine stages it through its pinned buffer (dev_api.cu: gpbdev_vecchia_set_y)
    y_page = np.ascontiguousarray(y.copy())
    yp_ptr = y_page.ctypes.data_as(C.POINTER(C.c_double))
    for _ in range(W):
        chk(lib.GPB_EvalNegLogLikelihood(mdl.handle, yp_ptr, cp_ptr, None, C.byref(negll)))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        chk(lib.GPB_EvalNegLogLikelihood(mdl.handle, yp_ptr, cp_ptr, None, C.byref(negll)))
    barrier()
    e2e_page_s = (time.perf_counter() - t0) / args.steps
    outputs["negll_e2e_pageable"] = np.array([negll.value])
    sampler.stop_flag = True; sampler.join(2)

    # max over ranks
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, e2e_page_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s, e2e_page_s = float(t[0]), float(t[1]), float(t[2])

    # Laplace-Vecchia (configs[4]); all ranks take part (probe columns are sharded), rank 0 reports
    laplace_res = None
    if args.laplace_n > 0:
        laplace_res = time_laplace(args.laplace_n, None, ncores, reps=2, barrier=barrier if world > 1 else None)

    # GPBoost iteration (configs[2]/[3] shape): all ranks take part — GP rows and histogram rows are both sharded
    gb = None
    if args.boost_n > 0:
        gb = time_gpboost(args.boost_n, 5, None, ncores, F=args.boost_features)
    # BASELINE configs[3]: n = 5e6, 100 features, Vecchia m = 30 + trees, row-sharded over 8 GPUs — run when the job has 8 ranks
    gb3 = None
    if (args.config3 == "auto" and world == 8) or args.config3 == "on":
        try:
            gb3 = time_gpboost(5000000, 3, None, ncores, F=100, f32=True)
        except Exception as e:
            sys.stderr.write("configs[3] measurement failed: %r\n" % (e,))

    dense_res = None
    if args.dense_n > 0 and world == 1:
        try:
            dense_res = time_dense(args.dense_n, None, ncores)
        except Exception as e:
            sys.stderr.write("dense measurement failed: %r\n" % (e,))
    gg = None
    if args.boost_n > 0 and world == 1:
        try:
            gg = time_gpboost_grouped(args.boost_n, 10, None, ncores, F=args.boost_features)
        except Exception as e:  # a secondary measurement must not cost the headline line
            sys.stderr.write("gpboost_grouped measurement failed: %r\n" % (e,))

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        rows_per_rank = (N_OBS + world - 1) // world
        achieved_gbs = ALGO_BYTES_PER_OBS * rows_per_rank / (dev_ms * 1e-3) / 1e9
        fp64_peak = C.c_double(0)
        lib.gpbdev_fp64_peak(local_rank, C.byref(fp64_peak))
        achieved_tf = ALGO_FLOPS_PER_OBS * rows_per_rank / (dev_ms * 1e-3) / 1e12
        line = {
            "metric": "gp_loglik_evals_per_sec", "value": 1e3 / dev_ms, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "cov_pars": COV_PARS.tolist(), "l2": "flushed (256 MiB write) before every timed pass",
                       "sharding": "rows of the ordered observations over %d rank(s); 9 fp64 sums all-reduced" % world,
                       "model_creation_s": t_create},
            "e2e": {"value": 1.0 / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": int(8 * N_OBS + 24), "d2h_bytes_per_step": 72 + 8,
                    "ms_per_step": e2e_s * 1e3, "call": "GPB_EvalNegLogLikelihood(handle, y_host_pinned, cov_pars, NULL, &negll)",
                    "pageable_y": {"value": 1.0 / e2e_page_s, "ms_per_step": e2e_page_s * 1e3,
                                   "note": "same call with y in ordinary numpy memory (staged through the engine's pinned buffer)"}},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                         "traffic": ncu_traffic_bytes() if world == 1 else None, "traffic_unit": "bytes per launch (ncu --set full, profiles/r02_ncu_raw_summary.txt)",
                         "kernel": "vecchia_nll2_kernel<MATERN15> (two observations per warp)", "kernel_ms": dev_ms,
                         "algorithmic_bytes_per_obs": ALGO_BYTES_PER_OBS, "peak_source": peak_src,
                         "note": "this kernel is FP64-pipe bound, not HBM bound (SURVEY §8d, DESIGN.md): see roofline_fp64"},
            "roofline_fp64": {"bound": "fp64_fma", "achieved": achieved_tf, "peak": fp64_peak.value, "unit": "TFLOP/s",
                              "frac": achieved_tf / fp64_peak.value if fp64_peak.value > 0 else None,
                              "flops_per_obs": ALGO_FLOPS_PER_OBS, "peak_source": "measured live: gpbdev_fp64_peak DFMA microbenchmark"},
            "negll": negll_value,
        }
        if gb is not None:
            line["gpboost"] = {"iters_per_sec": 1.0 / gb["sec_per_iter"], "ms_per_iter": gb["sec_per_iter"] * 1e3, "n": args.boost_n,
                               "first_iter_s": gb["first_iter_s"], "cov_pars": gb["cov_pars"],
                               "note": "LGBM_BoosterUpdateOneIter, GPBoost Vecchia m=30 + 31-leaf trees on n x 50 features, covariance "
                                       "parameters re-fitted every iteration (BASELINE metric (i)); host buffers, end to end"}
        if gb is not None and "hist_roofline" in gb:
            line["gpboost"]["roofline"] = gb["hist_roofline"]
        if gb3 is not None:
            line["gpboost_config3"] = {"iters_per_sec": 1.0 / gb3["sec_per_iter"], "ms_per_iter": gb3["sec_per_iter"] * 1e3, "n": 5000000, "features": 100,
                                       "first_iter_s": gb3["first_iter_s"], "cov_pars": gb3["cov_pars"], "roofline": gb3.get("hist_roofline"),
                                       "note": "BASELINE configs[3]: LGBM_BoosterUpdateOneIter, Vecchia m=30 + 31-leaf trees, n=5e6 x 100 float32 features, GP rows "
                                               "and histogram rows sharded over the ranks"}
        if dense_res is not None:
            line["dense"] = {"evals_per_sec": 1.0 / dense_res["sec_per_eval"], "n": args.dense_n, **dense_res,
                             "note": "GPB_EvalNegLogLikelihood / GPB_OptimCovPar, exact GP n x n dense Cholesky on the device (BASELINE configs[0])"}
        if gg is not None:
            line["gpboost_grouped"] = {"iters_per_sec": 1.0 / gg["grouped"]["sec_per_iter"], "ms_per_iter": gg["grouped"]["sec_per_iter"] * 1e3,
                                       "trees_only_ms_per_iter": gg["trees_only"]["sec_per_iter"] * 1e3, "n": args.boost_n,
                                       "first_iter_s": gg["grouped"]["first_iter_s"], "cov_pars": gg["grouped"]["cov_pars"],
                                       "roofline": gg["trees_only"].get("hist_roofline"),
                                       "note": "LGBM_BoosterUpdateOneIter, single-level grouped random effect (1e4 groups) + 31-leaf trees on "
                                               "n x 50 features (BASELINE configs[2]); trees_only = the same data without a random-effects model"}
        if laplace_res is not None:
            line["laplace"] = {"evals_per_sec": 1.0 / laplace_res["sec_per_eval"], **laplace_res,
                               "note": "GPB_EvalNegLogLikelihood, bernoulli_logit + latent Vecchia GP m=30 (BASELINE configs[4]); with N GPUs "
                                       "the 50 SLQ probe columns are sharded over the ranks (every rank holds the whole factor)"}
        if not args.no_cpu_baseline and world == 1:
            ns = args.cpu_sample_n
            res = time_reference(ns, 3, 1, ncores)
            if res is not None:
                v = 1.0 / (res["sec_per_eval"] * (N_OBS / ns))
                line["cpu_baseline"] = {"value": v, "unit": "evals/s", "cores": ncores, "kind": "reference",
                                        "sample": "n=%d sub-problem of the same workload, 3 timed GPB_EvalNegLogLikelihood calls of the "
                                                  "unmodified reference CPU library; per-eval time scaled linearly to n=1e6" % ns}
        if args.dump_outputs:
            if laplace_res is not None:
                outputs["laplace_negll"] = np.array([laplace_res["negll"]])
            if gb is not None:
                outputs["gpboost_cov_pars"] = np.array(gb["cov_pars"])
            if dense_res is not None:
                outputs["dense_negll"] = np.array([dense_res["negll"]])
                outputs["dense_fit_cov_pars"] = np.array(dense_res["fit_cov_pars"])
            if gg is not None:
                outputs["gpboost_grouped_cov_pars"] = np.array(gg["grouped"]["cov_pars"])
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(arr, dtype=np.float64))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    del cb_keep
    return 0


if __name__ == "__main__":
    sys.exit(main())
