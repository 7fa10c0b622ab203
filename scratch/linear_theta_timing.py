# -*- coding: utf-8 -*-
"""ms per sweep (one PSMFIter sweep + predict + Adam update) of theta learning with an affine dynamics callable:
marked with nonlinearities.affine (device linear dynamics, one launch per sweep) against the same callable unmarked
(external path, one launch, one host Jacobian and one PCIe round trip per step).

    python scratch/linear_theta_timing.py [--sweeps 5] [--d 20 2000]

Prints one JSON line per shape with the GPU name and power limit it ran on."""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from rpsmf_b200 import PSMFIter                      # noqa: E402
from rpsmf_b200.nonlinearities import affine          # noqa: E402


def _fn(r):
    B = 0.05 * np.random.RandomState(r).randn(r, r)

    def f(theta, x, t):
        th = theta.reshape(-1)
        return (0.85 * np.eye(r) + 0.1 * np.diag(np.sin(th)) + B) @ x + (0.2 * th * th).reshape(r, 1)
    return f


def _time(fn, d, r, T, sweeps, n_pred):
    rng = np.random.RandomState(0)
    C0 = rng.randn(d, r)
    Y = rng.randn(T, d)
    y = {k + 1: Y[k].reshape(d, 1) for k in range(T)}
    Q, R = 0.05 * np.eye(r), 2.0 * np.eye(d)
    o = PSMFIter(0.3 * np.ones((r, 1)), C0, 0.5 * np.eye(r), np.zeros((r, 1)), np.eye(r), {k: Q for k in range(T + 1)},
                 {k: R for k in range(T + 1)}, fn)
    o.optim_init(gam=1e-3)
    times = []
    for i in range(1, sweeps + 2):                    # sweep 1 warms up (engine creation, module load, first copies)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        o.step(y, i, T)
        o.predict(i, T, n_pred)
        o.optim_update(i)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    o.close()
    return 1e3 * float(np.median(times[1:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=5)
    ap.add_argument("--d", type=int, nargs="+", default=[20, 2000])
    ap.add_argument("--r", type=int, default=6)
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--n-pred", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except Exception:
        gpu = torch.cuda.get_device_name(0)
    for d in a.d:
        f = _fn(a.r)
        marked = _time(affine(f), d, a.r, a.T, a.sweeps, a.n_pred)
        unmarked = _time(f, d, a.r, a.T, a.sweeps, a.n_pred)
        print(json.dumps(dict(d=d, r=a.r, T=a.T, ms_per_sweep_marked=round(marked, 3), ms_per_sweep_unmarked=round(unmarked, 3),
                              speedup=round(unmarked / marked, 1), gpu=gpu)))


if __name__ == "__main__":
    main()
