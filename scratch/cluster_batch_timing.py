# -*- coding: utf-8 -*-
"""Series-steps per second of a batch of S independent series, three ways:
  (a) one single-series engine (automatic kernel) run once per series, one after another;
  (b) one engine of S series with one CTA per series (batch or direct-load kernel), where that fits;
  (c) one engine of S series with a thread-block cluster per series: the automatic size and ctas = 2, 4, 8, 16.

    python scratch/cluster_batch_timing.py [--launches 2] [--r 8 16] [--S 2 8 32 128] [--d 4000 20000 100000]

rPSMF, fp64, 20 % missing, one launch = 500 filter steps; one warm-up launch per arm, then CUDA events around `launches`
launches.  All series read the same Y / M (stride 0 over the series axis) so that S = 128 at d = 100 000 fits the device;
C and the state are per series.  Prints one JSON line per shape and a first line with the GPU name and power limit."""

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from rpsmf_b200 import FilterEngine                   # noqa: E402
from rpsmf_b200._capi import PsmfError                # noqa: E402
from synth import impute_init                         # noqa: E402

W = 500


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def _engine(d, r, S, C0, x0, **kw):
    init = impute_init(r)
    eng = FilterEngine(d, r, n_series=S, robust=True, **kw)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    return eng


def _time(launch, launches):
    launch()                                           # warm-up
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(launches):
        launch()
    ev[1].record()
    ev[1].synchronize()
    return ev[0].elapsed_time(ev[1]) / 1e3 / launches  # seconds per launch of W steps (of every series)


def shape(d, r, S, launches, dev):
    g = torch.Generator(device="cpu").manual_seed(d + r)
    Y1 = torch.randn((1, W, d), generator=g, dtype=torch.float64).to(dev)
    M1 = (torch.rand((1, W, d), generator=g) >= 0.2).to(torch.uint8).to(dev)
    Y1 = Y1 * M1
    C0 = torch.rand((S, d, r), generator=g, dtype=torch.float64)
    x0 = torch.rand((S, r), generator=g, dtype=torch.float64)
    out = dict(d=d, r=r, S=S)

    # (a) one engine per series, one after another (one engine reused: the same launches)
    eng = _engine(d, r, 1, C0[0], x0[0])
    t = _time(lambda: [eng.run(Y1, M1, want_X=False) for _ in range(S)], launches)
    info = eng.launch_info()
    assert eng.status() == -1
    eng.close()
    out["a_sequential"] = dict(series_steps_per_s=S * W / t, kernel=info["kernel"], ctas=info["ctas"])

    Y, M = Y1.expand(S, W, d), M1.expand(S, W, d)
    # the automatic engine is (b) while one CTA per series fits, else (c) at the automatic size
    for name, ctas in [("auto", 0)] + [("c_%d" % c, c) for c in (2, 4, 8, 16)]:
        try:
            eng = _engine(d, r, S, C0, x0, ctas=ctas)
        except PsmfError as e:
            out[name] = "refused: " + str(e)
            continue
        t = _time(lambda: eng.run(Y, M, want_X=False), launches)
        info = eng.launch_info()
        assert eng.status() == -1
        eng.close()
        rec = dict(series_steps_per_s=S * W / t, kernel=info["kernel"], ctas=info["ctas"])
        if name == "auto":
            one = info["ctas"] == 1
            out["b_one_cta"] = rec if one else "not available: one CTA per series does not fit"
            out["c_auto"] = "not selected: one CTA per series fits" if one else rec
        else:
            out[name] = rec
    del Y1, M1
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=2)
    ap.add_argument("--r", type=int, nargs="+", default=[8, 16])
    ap.add_argument("--S", type=int, nargs="+", default=[2, 8, 32, 128])
    ap.add_argument("--d", type=int, nargs="+", default=[4000, 20000, 100000])
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    print(json.dumps(dict(gpu=_gpu(), steps_per_launch=W, launches=a.launches)), flush=True)
    for r in a.r:
        for S in a.S:
            for d in a.d:
                print(json.dumps(shape(d, r, S, a.launches, dev)), flush=True)


if __name__ == "__main__":
    main()
