"""Throughput of the MLP training path (mCaller --train -c NN) on seeded rows: the GPU fit of one job alone and of the 12
jobs of a `-b A` run together (two model keys x (5 cross-validation folds of 80 % + 1 final fit)), the host's time drawing
the sample orders and the part of it the GPU waited for, and scikit-learn's own time per epoch on the same host.
Prints one JSON line per size, with the card's name and power limit read in the same run.

    python tools/train_throughput.py --rows 300000 3000000 [--sklearn-epochs 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _rows(n, seed, d=7):
    rng = np.random.RandomState(seed)
    x = rng.normal(size=(n, d))
    y = (x[:, 0] - 0.5 * x[:, 1] + rng.normal(size=n) > 0).astype(np.float64)
    return x, y


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[300000, 3000000], help="rows per model key")
    ap.add_argument("--sklearn-epochs", type=int, default=3, help="epochs of the scikit-learn timing (at the first size)")
    a = ap.parse_args()
    import torch
    from mcaller_b200 import build, train as tr
    build.build()
    card = _card()
    tr.fit_mlp_jobs(*_rows(1000, 0), [(np.arange(1000), 0)])          # module load, first launch
    for n in a.rows:
        xs, ys = zip(*(_rows(n, 10 + key) for key in range(2)))
        x, y = np.concatenate(xs), np.concatenate(ys)
        jobs = []
        for key in range(2):
            base = key * n
            folds = np.array_split(np.random.RandomState(key).permutation(n), 5)
            for f in range(5):
                jobs.append((base + np.sort(np.concatenate(folds[:f] + folds[f + 1:])), 0))
            jobs.append((base + np.arange(n), 0))
        res = {"rows_per_key": n, "jobs": len(jobs), "card": card}
        st = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        one = tr.fit_mlp_jobs(x, y, [jobs[5]], stats=st)
        torch.cuda.synchronize()
        res["one_job_s"] = time.perf_counter() - t0
        res["one_job_epochs"] = one[0][1]
        res["one_job_draw_s"], res["one_job_gpu_waited_s"] = st["draw_s"], st["wait_s"]
        st = {}
        t0 = time.perf_counter()
        all12 = tr.fit_mlp_jobs(x, y, jobs, stats=st)
        torch.cuda.synchronize()
        res["all_jobs_s"] = time.perf_counter() - t0
        res["all_jobs_epochs"] = [r[1] for r in all12]
        res["all_jobs_draw_s"], res["all_jobs_gpu_waited_s"] = st["draw_s"], st["wait_s"]
        res["one_job_s_per_epoch"] = res["one_job_s"] / max(1, res["one_job_epochs"])
        if n == a.rows[0] and a.sklearn_epochs > 0:
            from sklearn.neural_network import MLPClassifier
            params = dict(tr.SHIPPED_NN, max_iter=a.sklearn_epochs)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                t0 = time.perf_counter()
                MLPClassifier(random_state=0, **params).fit(x[:n], y[:n])
                res["sklearn_s_per_epoch"] = (time.perf_counter() - t0) / a.sklearn_epochs
            res["sklearn_cpu_threads"] = os.cpu_count()
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
