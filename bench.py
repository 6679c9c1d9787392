#!/usr/bin/env python
"""bench.py -- candidate-fits/sec of DistGridSearchCV(LogisticRegression) on synthetic
1M x 256 fp32, 512-point C grid x 5 folds (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU path
    python bench.py --config {3,4,5} ...                           # the other BASELINE.json configs (bench_configs.py)

A "step" is one complete pass of the hot path: every (candidate, fold) column fitted with
the batched L-BFGS solver and scored on its held-out rows.  `value` is measured with
(X, y, folds) already resident in HBM; `e2e` goes through the public drop-in API
(DistGridSearchCV.fit on HOST numpy arrays: H2D staging, fits, scoring, D2H of results; refit
excluded as SURVEY.md section 8d defines the metric).  Under torchrun (N > 1) columns are dealt
round-robin to ranks ("weak": the per-rank batch shrinks, total work is fixed -> "strong").
One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "candidate-fits/sec (params x folds) DistGridSearchCV LogReg 1Mx256"
UNIT = "fits/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                   help="BASELINE.json configs[k - 1]: 2 = the headline (default), 3 OvR-SGD, 4 forest, 5 Ridge search + predict "
                        "(bench_configs.py)")
    p.add_argument("--n", type=int, default=0, help="rows (0 = the config's size)")
    p.add_argument("--d", type=int, default=0, help="features (0 = the config's size)")
    p.add_argument("--candidates", type=int, default=512)
    p.add_argument("--folds", type=int, default=5)
    p.add_argument("--cpu-sample", type=int, default=40, help="fits timed for cpu_baseline / compared for parity (0 = skip)")
    p.add_argument("--kernel", type=int, default=0, help="0 auto, 1 SIMT fp32, 2 tcgen05")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and (a.config != 2 or a.impl != "b200"):
        p.error("--dump-outputs writes the outputs of the headline workload's CUDA path (--config 2 --impl b200)")
    if a.config == 2:
        a.n = a.n or 1_000_000
        a.d = a.d or 256
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        j = json.load(open(path))
        return {"bf16_burst": j["bf16_tflops"], "bf16_sustained": j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                "hbm": j["hbm_gbs"], "src": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None
        self.t0 = self.t1 = None

    # nvidia-smi takes driver locks while it starts up (hundreds of ms of stalled CUDA calls), so it
    # is started before the warm-up; only samples taken between begin() and end() are reported.
    def begin(self):
        self.t0 = time.monotonic()

    def end(self):
        self.t1 = time.monotonic()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "250"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if (self.t0 is None or t >= self.t0) and (self.t1 is None or t <= self.t1 + 0.25)]
        if not rows:
            rows = [r for _, r in self.rows[-1:]]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_tasks(n_cands, n_folds, n_fits):
    """The bounded sample of (candidate, fold) tasks the CPU legs run: whole candidates (every fold of
    a C value, so that mean_test_score of the sub-grid is comparable), C spread evenly over the grid."""
    n_c = max(1, n_fits // n_folds)
    idx = np.unique(np.linspace(0, n_cands - 1, n_c).round().astype(int))
    tasks = [(int(ci), f) for ci in idx for f in range(n_folds)]
    if n_fits < n_folds:
        tasks = tasks[:n_fits]
    return tasks


def cpu_fits_per_sec(X, y, fold, Cs, tasks, n_jobs=None):
    """The reference's sc=None branch (search.py:388-409): the same per-task function
    (oracle.search_oracle.fit_and_score <- search.py:180-288) fanned out with joblib over the host
    cores, on a bounded sample of (candidate, fold) tasks of the same workload.  ONE wave of
    n_jobs = min(len(tasks), 40, cores) worker processes, each with cores // n_jobs BLAS threads (the
    fastest way found to use the box: a single process with all BLAS threads is limited by one
    sgemv stream; 8 x 16 threads measured 0.12-0.40 fits/s, 32 x 4 threads the same or better).
    Thread counts are set explicitly (torchrun exports OMP_NUM_THREADS=1).
    Returns (fits/s, seconds, scores aligned with tasks, n_jobs, inner_threads)."""
    from joblib import Parallel, delayed, parallel_config
    from sklearn.linear_model import LogisticRegression
    from sklearn.metrics import check_scoring
    from threadpoolctl import threadpool_limits
    from oracle.search_oracle import fit_and_score
    est = LogisticRegression()
    scorer = check_scoring(est)
    cores = os.cpu_count() or 1
    if n_jobs is None:
        n_jobs = max(1, min(len(tasks), 40, cores))
    inner = max(1, cores // n_jobs)
    jobs = [({"C": float(Cs[ci])}, np.flatnonzero(fold != f), np.flatnonzero(fold == f)) for ci, f in tasks]
    import warnings
    t0 = time.time()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if n_jobs == 1:
            with threadpool_limits(limits=inner):
                out = [fit_and_score(est, X, y, scorer, tr, te, p) for p, tr, te in jobs]
        else:
            with parallel_config(backend="loky", n_jobs=n_jobs, inner_max_num_threads=inner):
                out = Parallel()(delayed(fit_and_score)(est, X, y, scorer, tr, te, p) for p, tr, te in jobs)
    dt = time.time() - t0
    return len(jobs) / dt, dt, [o[0]["score"] for o in out], n_jobs, inner


def parity_block(cv_results, tasks, cpu_scores, fold, Cs, n_folds):
    """The CPU leg's scores (the reference's per-task function on the exact bench inputs) against the
    device search's cv_results_ at the same (candidate, fold): the checker of the headline workload."""
    n_test = np.bincount(fold.astype(np.int64), minlength=n_folds)
    flips, dsc = [], []
    by_c = {}
    for (ci, f), sc in zip(tasks, cpu_scores):
        g = float(cv_results["split%d_test_score" % f][ci])
        flips.append(abs(int(round(g * n_test[f])) - int(round(sc * n_test[f]))))
        dsc.append(abs(g - sc))
        by_c.setdefault(ci, {})[f] = (sc, g)
    full = sorted(ci for ci, v in by_c.items() if len(v) == n_folds)
    out = {"n_compared": len(tasks), "max_flips_per_fold": int(max(flips)), "mean_flips_per_fold": float(np.mean(flips)),
           "test_rows_per_fold": int(n_test.min()), "max_abs_dscore_split": float(max(dsc)),
           "checker": "oracle.search_oracle.fit_and_score (ref search.py:180-288) on the same inputs"}
    if full:
        w = n_test / n_test.sum()      # iid weighting by test-fold size (ref search.py:509-519)
        cpu_mean = np.array([sum(w[f] * by_c[ci][f][0] for f in range(n_folds)) for ci in full])
        gpu_mean = np.array([float(cv_results["mean_test_score"][ci]) for ci in full])
        out.update(subgrid_C=[float(Cs[ci]) for ci in full],
                   max_abs_dscore=float(np.max(np.abs(cpu_mean - gpu_mean))),
                   max_rel_dscore=float(np.max(np.abs(cpu_mean - gpu_mean) / np.abs(cpu_mean))),
                   best_C_cpu_on_subgrid=float(Cs[full[int(np.argmax(cpu_mean))]]),
                   best_C_gpu_on_subgrid=float(Cs[full[int(np.argmax(gpu_mean))]]),
                   best_C_equal_on_subgrid=bool(int(np.argmax(cpu_mean)) == int(np.argmax(gpu_mean))),
                   cpu_best_margin=float(np.sort(cpu_mean)[-1] - np.sort(cpu_mean)[-2]) if len(full) > 1 else None,
                   # how much worse, by the CPU leg's own scores, the device's choice is than the CPU's: a value
                   # below the CPU-vs-device differences above means the two picked from a tie
                   cpu_score_of_device_choice_minus_cpu_best=float(cpu_mean[int(np.argmax(gpu_mean))] - cpu_mean.max()),
                   best_C_tied=bool(cpu_mean.max() - cpu_mean[int(np.argmax(gpu_mean))]
                                    <= max(2e-5, float(np.max(np.abs(cpu_mean - gpu_mean))))),
                   cpu_mean_test_score=[float(v) for v in cpu_mean], device_mean_test_score=[float(v) for v in gpu_mean])
    return out


def fold_ids(y, n_folds):
    from sklearn.model_selection import StratifiedKFold
    fold = np.zeros(len(y), np.int8)
    for k, (_, te) in enumerate(StratifiedKFold(n_folds).split(np.zeros((len(y), 1)), y)):
        fold[te] = k
    return fold


DUMP_LIMIT = 63 * 10 ** 6      # array bytes; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, res, correct, count, n_cols, rank, world, order, cost):
    """--dump-outputs: the arrays one timed step returns (logreg_fit_batch's coef / n_iter / status / loss /
    n_evals, linear_score_batch's correct / count), one row per (candidate, fold) column in candidate-major
    order (column = candidate * folds + fold) whatever the dealing over ranks, written by rank 0 as
    float32 / float64 .npy files.  column.npy lists the columns written: all of them, or, when they would
    exceed 64 MB, a fixed seeded sample, so that two builds run with the same arguments compare row for row."""
    from skdist_b200 import parallel
    local = {"coef": res["coef"], "n_iter": res["n_iter"], "status": res["status"], "loss": res["loss"],
             "n_evals": res["n_evals"], "correct": correct, "count": count}
    full = {k: parallel.all_gather_blocks(v, n_cols, rank, world, order, cost=cost) for k, v in local.items()}
    if rank != 0:
        return
    full = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in full.items()}
    row_bytes = 8 + sum(v[0].nbytes for v in full.values())
    cols = np.arange(n_cols)
    if row_bytes * n_cols > DUMP_LIMIT:
        cols = np.sort(np.random.default_rng(0).choice(n_cols, DUMP_LIMIT // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "column.npy"), cols.astype(np.float64))
    for k, v in full.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[cols])


def workload_name(a):
    return "DistGridSearchCV(LogisticRegression) %d-point C grid x %d folds, synthetic G1 %dx%d fp32" % (
        a.candidates, a.folds, a.n, a.d)


def run_reference(a):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from skdist_b200.datasets import make_g1_classification
    X, y = make_g1_classification(a.n, a.d, seed=0)
    fold = fold_ids(y, a.folds)
    Cs = np.logspace(-4, 4, a.candidates)
    cores = os.cpu_count() or 1
    # The K timed steps are K equal bounded samples of the workload (each a few (candidate, fold) fits,
    # C spread over the grid).  All K samples are run as ONE wave of worker processes that uses every
    # host core (about 32-40 workers x 3-4 BLAS threads), whatever --steps is: the step time reported
    # is the wave time / K.  (Round 1 ran 2 fits x 64 threads per step when --steps was large, the
    # slowest way to use the box.)
    st = max(1, a.n // 20000)              # warm-up: page the data in with one short fit on a strided subsample
    for _ in range(min(a.warmup, 1)):
        cpu_fits_per_sec(np.ascontiguousarray(X[::st]), y[::st], fold[::st], Cs, [(len(Cs) // 2, 0)])
    per_step = max(1, int(round(max(a.cpu_sample, 32) / max(1, a.steps))))
    tasks = cpu_tasks(a.candidates, a.folds, per_step * a.steps)[:per_step * a.steps]
    while len(tasks) < per_step * a.steps:      # tiny grids: cycle
        tasks = tasks + tasks[:per_step * a.steps - len(tasks)]
    v, tot_t, _, nj, inner = cpu_fits_per_sec(X, y, fold, Cs, tasks)
    tot_fits = len(tasks)
    value = tot_fits / tot_t
    vals = [None] * a.steps
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / max(1, len(vals)),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": workload_name(a), "inputs": "exceed L2"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d (candidate, fold) fits per step x %d steps run as one wave, C spread over the grid, joblib "
                                   "n_jobs=%d x %d BLAS threads (reference sc=None branch, search.py:388-409)"
                                   % (per_step, a.steps, nj, inner)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    a = parse()
    if a.config != 2:
        import bench_configs
        if a.impl == "reference":
            return bench_configs.run_reference(a)
        return bench_configs.run(a, ClockSampler, peaks)
    if a.impl == "reference":
        return run_reference(a)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from sklearn.linear_model import LogisticRegression
    from skdist.distribute.search import DistGridSearchCV
    from skdist_b200 import parallel
    from skdist_b200.datasets import make_g1_classification
    from skdist_b200.engine import get_engine

    X, y = make_g1_classification(a.n, a.d, seed=0)   # every rank builds the same seeded inputs
    Cs = np.logspace(-4, 4, a.candidates)
    fold = fold_ids(y, a.folds)
    eng = get_engine()
    if a.kernel:
        eng.set_kernel(a.kernel)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: inputs staged once, each step = fit + score of this rank's columns
    eng.stage_x(X)
    eng.stage_labels(y.astype(np.int32))
    eng.stage_folds(fold, a.folds)
    n_cols = a.candidates * a.folds
    # same dealing as DistGridSearchCV: blocks of 128 consecutive candidates of one fold per rank
    deal_order = (np.arange(a.candidates)[None, :] * a.folds + np.arange(a.folds)[:, None]).ravel()
    col_cost = np.repeat(parallel.logreg_column_cost(Cs), a.folds) if world > 1 else None
    my = parallel.shard_blocks(n_cols, rank, world, deal_order, cost=col_cost)
    C_cols = np.repeat(Cs, a.folds)[my]
    f_cols = np.tile(np.arange(a.folds, dtype=np.int32), a.candidates)[my]
    pos = np.ones(len(my), np.int32)

    def step():
        res = eng.logreg_fit_batch(C_cols, f_cols, pos)
        correct, count = eng.linear_score_batch(res["coef"], f_cols, pos)
        return res, correct, count

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(a.warmup):
        step()
    barrier()
    sampler.begin()
    eng.profile(1)
    c0 = eng.counters()
    # CUDA events on the stream the kernels are launched on (the library's own stream;
    # torch.cuda.Event would only see torch's current stream)
    eng.timer_start()
    for _ in range(a.steps):
        res, correct, count = step()
    wall = eng.timer_stop()
    barrier()
    sampler.end()
    prof = eng.profile(0)
    c1 = eng.counters()
    clocks = sampler.stop() if rank == 0 else None
    # device time between the two events, max over ranks
    tt = torch.tensor([wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_steps = float(tt.item())
    value = n_cols * a.steps / t_steps
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, res, correct, count, n_cols, rank, world, deal_order, col_cost)

    # ---- end-to-end arm: public API on host arrays (H2D + fits + scoring + D2H), refit excluded
    gs_times = []
    h2d = d2h = 0
    E2E_REPS = 3
    for i in range(1 + E2E_REPS):   # one warm-up, then E2E_REPS timed fits (the median is reported)
        barrier()
        cc0 = eng.counters()
        t0 = time.perf_counter()
        gs = DistGridSearchCV(LogisticRegression(), {"C": list(Cs)}, None, cv=a.folds, refit=False)
        gs.fit(X, y)
        barrier()
        gs_times.append(time.perf_counter() - t0)
        cc1 = eng.counters()
        h2d, d2h = cc1["h2d_bytes"] - cc0["h2d_bytes"], cc1["d2h_bytes"] - cc0["d2h_bytes"]
    te = torch.tensor(gs_times[1:], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)      # per repetition: the slowest rank
    e2e_all = sorted(float(v) for v in te.tolist())
    e2e_seconds = e2e_all[len(e2e_all) // 2]
    e2e_value = n_cols / e2e_seconds

    if rank == 0:
        pk = peaks()
        achieved = prof["eval_flops"] / (prof["eval_ms"] * 1e-3) / 1e12 if prof["eval_ms"] > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * t_steps / a.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a), "inputs": "exceed L2 (X is %.2f GB)" % (X.nbytes / 1e9),
                       "parallelism": "blocks of 128 same-fold columns dealt over %d rank(s) (longest first, by C), X replicated" % world,
                       "kernel": {0: "auto", 1: "simt-fp32", 2: "tcgen05"}[a.kernel],
                       "mean_test_score_best": float(np.max(gs.cv_results_["mean_test_score"])),
                       "best_C": float(gs.best_params_["C"]),
                       "rounds_per_step": prof["rounds"] / max(1, a.steps)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "seconds": e2e_seconds,
                    "seconds_all": e2e_all, "reported": "median of %d timed fits after one warm-up" % E2E_REPS},
            "gpu_launches": int(c1["launches"] - c0["launches"]),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["bf16_sustained"],
                         "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"], "traffic": None,
                         "peak_source": pk["src"] + " bf16 dense (sustained)",
                         "kernel": "logistic loss+gradient evaluation (rank 0)",
                         "launches": prof["eval_launches"], "avg_launch_ms": prof["eval_ms"] / max(1, prof["eval_launches"]),
                         "algorithmic_flops": "4 * n_train * d per active column per launch",
                         # fp32-grade accuracy costs 3 fp16 MMA passes per algorithmic FLOP
                         "mma_passes": 3, "tensor_issue_frac": 3 * achieved / pk["bf16_sustained"]},
        }
        # DRAM traffic of the dominant kernel comes from the committed ncu capture (bench.py never runs
        # under a profiler); only reported for the workload it was captured on
        tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "roofline_traffic.json")
        if os.path.exists(tpath) and (a.n, a.d, a.candidates, a.folds, a.kernel) == (1_000_000, 256, 512, 5, 0):
            with open(tpath) as f:
                tj = json.load(f)
            line["roofline"]["traffic"] = tj["dram_bytes_per_launch"]
            line["roofline"]["traffic_source"] = tj["source"]
        if world == 1 and a.cpu_sample > 0:
            cores = os.cpu_count() or 1
            tasks = cpu_tasks(a.candidates, a.folds, a.cpu_sample)
            v, dt, cpu_scores, nj, inner = cpu_fits_per_sec(X, y, fold, Cs, tasks)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d (candidate, fold) fits of the same workload in %.1f s (one wave), whole candidates, C spread "
                          "over the grid, joblib n_jobs=%d x %d BLAS threads (reference sc=None branch, search.py:388-409)"
                          % (len(tasks), dt, nj, inner)}
            line["parity"] = parity_block(gs.cv_results_, tasks, cpu_scores, fold, Cs, a.folds)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
