# -*- coding: utf-8 -*-
"""Cost of PSMF_LOGLIK: ms per launch of bench.py's workloads L and B with the flag off and on, in alternating rounds.

    python scratch/loglik_timing.py [--rounds 5] [--launches 4] [--T 2000]

Workload L: one rPSMF series, d = 1,000,000, r = 16, fp64, 20 % missing, one launch = 500 filter steps on the TMA-staged
kernel, the per-step scalar record written in both arms (8 wide without the flag, 10 wide with it).  Workload B: 4096
series of d = 512, r = 8, one launch = 500 steps on the batch kernel; without the flag no record, with it the 10-wide one.
The inputs are bench.py's (bench_data.py), over a shorter horizon T.  Prints one JSON line with the GPU name and power limit."""

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import bench_data as bd                               # noqa: E402
from rpsmf_b200 import FilterEngine                   # noqa: E402


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def _arm(Y, M, C0, x0, init, S, loglik, W, want_scal, **kw):
    d, r = Y.shape[-1], C0.shape[-1]
    eng = FilterEngine(d, r, n_series=S, robust=True, loglik=loglik, **kw)
    T = Y.shape[-2]
    sc = torch.empty((S, W, 10 if loglik else 8), dtype=torch.float64, device=Y.device) if want_scal else None

    def launch(i):
        w = i % (T // W)
        sl = slice(w * W, (w + 1) * W)
        eng.run(Y[..., sl, :], M[..., sl, :], k0=1 + i * W, want_X=False, scal_out=sc)

    def reset():
        eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    return eng, launch, reset


def _time(arm, launches):
    eng, launch, reset = arm
    reset()
    launch(0)                                          # warm-up
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for i in range(launches):
        launch(1 + i)
    ev[1].record()
    ev[1].synchronize()
    assert eng.status() == -1
    return ev[0].elapsed_time(ev[1]) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=4)
    ap.add_argument("--T", type=int, default=2000)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    W = 500
    out = dict(gpu=_gpu(), window=W)
    init = bd.init_state(16)
    Y, M, C0, x0 = bd.make_series(torch, dev, 1_000_000, 0, 1_000_000, 16, a.T, torch.float64)
    arms = {f: _arm(Y, M, C0, x0, init, 1, f, W, True, kernel=2) for f in (False, True)}
    res = {False: [], True: []}
    for _ in range(a.rounds):
        for f in (False, True):
            res[f].append(_time(arms[f], a.launches))
    assert all(arms[f][0].launch_info()["kernel"] == "tma" for f in arms)
    out["L_ms_per_launch"] = {"off": res[False], "on": res[True]}
    for f in arms:
        arms[f][0].close()
    del Y, M, C0, x0, arms
    torch.cuda.empty_cache()
    init = bd.init_state(8)
    Y, M, C0, x0 = bd.make_batch(torch, dev, 0, 4096, 4096, 512, 8, min(a.T, 1000), torch.float64)
    arms = {f: _arm(Y, M, C0, x0, init, 4096, f, W, f) for f in (False, True)}
    res = {False: [], True: []}
    for _ in range(a.rounds):
        for f in (False, True):
            res[f].append(_time(arms[f], a.launches))
    assert all(arms[f][0].launch_info()["kernel"] == "batch" for f in arms)
    out["B_ms_per_launch"] = {"off": res[False], "on": res[True]}
    for f in arms:
        arms[f][0].close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
