# -*- coding: utf-8 -*-
"""Cost of the moment record and of the fixed-interval smoother on one GPU.

  forward   ms per launch with and without a moment buffer, alternating rounds in one process:
            workload L shape (d = 1M, r = 16, fp64, TMA-staged kernel, 500 steps) and workload B shape (512 series, d = 512,
            r = 8, batch kernel, 500 steps)
  smooth    ms per psmf_smooth call, with and without Ps_out: S = 1, T = 4393, r = 16 and S = 512, T = 500, r = 8
  pm25      Efull against EfullSmooth of rPSMF / PSMF on the stored PM25 30 % repeat (tests/golden/impute_pm25_30.npz), and
            over 100 repeats drawn as run_impute_experiment(batched=True) draws them (seed 1, the experiment's defaults),
            filtered side by side by fit_repeats(smooth=True)

Prints one JSON line per measurement, the GPU name and its power limit first.  Usage: python scratch/smooth_timing.py"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from rpsmf_b200 import FilterEngine, _capi  # noqa: E402


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=q)


def timed(fn, reps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / reps


def engine(d, r, S, kernel, ctas=0):
    eng = FilterEngine(d, r, n_series=S, kernel=kernel, ctas=ctas, robust=True)
    eng.set_state(C_=torch.randn(S, d, r, dtype=torch.float64, device="cuda") * 0.1, V=2 * np.eye(r), P=np.eye(r), x=np.zeros(r),
                  Q=0.1 * np.eye(r), rho=[10.0], lam=[1.8])
    return eng


def forward(name, d, r, S, T, kernel, rounds=5, reps=3):
    eng = engine(d, r, S, kernel)
    Y = torch.randn(S, T, d, dtype=torch.float64, device="cuda")
    X = torch.empty(S, T, r, dtype=torch.float64, device="cuda")
    mom = torch.empty(S, T, _capi.NMOM(r), dtype=torch.float64, device="cuda")
    off = lambda: eng.run(Y, None, X_out=X, want_X=False)
    on = lambda: eng.run(Y, None, X_out=X, want_X=False, moments_out=mom)
    off(); on()
    torch.cuda.synchronize()
    ms_off, ms_on = [], []
    for _ in range(rounds):
        ms_off.append(timed(off, reps))
        ms_on.append(timed(on, reps))
    info = eng.launch_info()
    eng.close()
    print(json.dumps(dict(what="forward", shape=name, d=d, r=r, S=S, T=T, kernel=info["kernel"], ms_off=ms_off, ms_on=ms_on,
                          median_off=float(np.median(ms_off)), median_on=float(np.median(ms_on)))), flush=True)


def smooth(S, T, r, reps=10):
    eng = engine(64, r, S, 1 if S == 1 else 3)
    Y = torch.randn(S, T, 64, dtype=torch.float64, device="cuda")
    out = eng.run(Y, None, want_X=False, want_moments=True)
    mom = out["moments"] if S > 1 else out["moments"].unsqueeze(0)
    eng.smooth(mom); eng.smooth(mom, want_P=True)
    res = dict(what="smooth", S=S, T=T, r=r, ms_X=timed(lambda: eng.smooth(mom), reps), ms_XP=timed(lambda: eng.smooth(mom, want_P=True), reps))
    eng.close()
    print(json.dumps(res), flush=True)


def pm25():
    from conftest import impute_case, load_golden
    from rpsmf_b200 import ProbabilisticSequentialMatrixFactorizer, robust_PSMF
    g = load_golden("impute_pm25_30")
    c = impute_case(g)
    r = c["r"]
    d, n = c["Y"].shape
    V, Q, R, P = 2 * np.eye(r), 0.1 * np.eye(r), 10 * np.eye(d), np.eye(r)
    for method in ("rPSMF", "PSMF"):
        Einit = float(g["rep0_%s_Einit" % method])
        X = c["X0"].copy()
        if method == "rPSMF":
            ep, ef, _, ib, efs = robust_PSMF(c["Y"], c["C0"].copy(), X, d, n, r, c["M"], c["Mmiss"], V, Q, R, P, 1.8, 2, c["Iter"],
                                             c["YorigInt"], Einit, smooth=True)
        else:
            ep, ef, _, ib, efs = ProbabilisticSequentialMatrixFactorizer(c["Y"], c["C0"].copy(), X, d, n, r, c["M"], c["Mmiss"], 0, V, Q, R,
                                                                         P, 2, c["Iter"], c["YorigInt"], Einit, smooth=True)
        print(json.dumps(dict(what="pm25_rep0", method=method, Epred=ep.tolist(), Efull=ef.tolist(), EfullSmooth=efs.tolist())), flush=True)


def pm25_repeats(repeats=100, seed=1):
    from conftest import load_golden
    from rpsmf_b200.experiment import DEFAULTS, prepare_missing, rmsem
    from rpsmf_b200.impute import fit_repeats
    hp = DEFAULTS
    Yorig = load_golden("impute_pm25_30")["Yorig"]
    YorigInt = np.nan_to_num(Yorig, nan=0.0)
    d, n = Yorig.shape
    r = hp["r"]
    for method in ("rPSMF", "PSMF"):
        np.random.seed(seed)
        Ys, Cs, Xs, Ms, Mms, Eis = [], [], [], [], [], []
        for _ in range(repeats):
            Ymiss = np.copy(Yorig)
            _, mm = prepare_missing(Ymiss, 0.30)
            M = np.array(np.invert(np.isnan(Ymiss)), dtype=int)
            Y = np.nan_to_num(Ymiss, nan=0.0)
            C = np.random.rand(d, r)
            X = np.random.rand(r, n)
            Ys.append(Y); Cs.append(C); Xs.append(X); Ms.append(M); Mms.append(mm); Eis.append(rmsem(C @ X, YorigInt, mm))
        _, ef, _, _, efs = fit_repeats(Ys, Cs, Xs, Ms, Mms, hp["v"] * np.eye(r), hp["q"] * np.eye(r), hp["rho"] * np.eye(d),
                                       hp["p"] * np.eye(r), hp["lambda0"], hp["sig"], hp["Iter"], YorigInt, Eis,
                                       robust=method == "rPSMF", smooth=True)
        a = np.array([e[0, -1] for e in ef]); b = np.array([e[0, -1] for e in efs])
        ok = np.isfinite(a) & np.isfinite(b)
        print(json.dumps(dict(what="pm25_100_repeats", method=method, seed=seed, finite=int(ok.sum()), Efull_mean=float(a[ok].mean()),
                              EfullSmooth_mean=float(b[ok].mean()), Efull_median=float(np.median(a[ok])),
                              EfullSmooth_median=float(np.median(b[ok])), smooth_lower=int(np.sum(b[ok] < a[ok])))), flush=True)


if __name__ == "__main__":
    print(json.dumps(gpu_line()), flush=True)
    forward("L", 1 << 20, 16, 1, 500, 2)
    forward("B", 512, 8, 512, 500, 3)
    smooth(1, 4393, 16)
    smooth(512, 500, 8)
    pm25()
    pm25_repeats()
