# -*- coding: utf-8 -*-
"""Drop-in replacements for the two flat model functions of the imputation experiment.

    robust_PSMF                                  ExperimentImpute/rPSMF.py:39-148
    ProbabilisticSequentialMatrixFactorizer      ExperimentImpute/PSMF.py:39-95

Same positional signatures, same return tuple ``(Epred, Efull, RunTime, InsideBars)``,
same side effect (``X`` is overwritten in place with the filtered x_t, rPSMF.py:104;
``C`` is left untouched).  The per-timestep loop bodies (rPSMF.py:81-135, PSMF.py:60-84)
run on the GPU through libpsmf_b200.so; the d x d temporaries of the reference are gone.

``smooth=True`` (keyword-only, also for ``fit_repeats``) adds one more returned value, ``EfullSmooth``, shaped like
``Efull``: the RMSE over Mmiss of C_T X^s per sweep, where X^s are the fixed-interval (RTS) smoothed states of the sweep
(include/psmf_b200.h psmf_smooth).  Every imputation here is offline -- the whole (d, n) matrix is on the device before
the first step -- so the state behind entry (i, t) may use the data after t as well.  ``X`` is still overwritten with
the filtered states.
"""

from __future__ import annotations

import time

import numpy as np
import torch

from . import _capi
from .engine import FilterEngine, ingest, transpose_mask


def _uniform_diag(R, d, name):
    """diag(R) for the CUDA path: a float when R = rho * I (every experiment of the reference), else the (d,) vector of a
    non-uniform diagonal R (PSMF_RHO_VECTOR).  Non-diagonal R is rejected -- the reference itself assumes a diagonal
    (rPSMF.py:91 inverts it entry by entry)."""
    R = np.asarray(R, dtype=np.float64)
    if R.ndim == 0:
        return float(R)
    if R.shape == (d,):
        dg = R
    elif R.shape == (d, d):
        dg = np.diagonal(R)
        if np.count_nonzero(R - np.diag(dg)) != 0:
            raise NotImplementedError("%s must be diagonal (the reference itself assumes this, rPSMF.py:91)" % name)
    else:
        raise ValueError("%s must be (d, d)" % name)
    if np.all(dg == dg[0]):
        return float(dg[0])
    return np.ascontiguousarray(dg, dtype=np.float64)


def _fit(Y, C, X, d, n, r, M, Mmiss, V, Q0, R0, P, lambda0, sig, Iter, YorigInt, Einit, robust, device=None,
         dtype=torch.float64, return_details=False, smooth=False):
    Y = np.asarray(Y); M = np.asarray(M)
    if Y.shape != (d, n) or M.shape != (d, n):
        raise ValueError("Y and M must be (d, n)")
    if X.shape != (r, n) or np.asarray(C).shape != (d, r):
        raise ValueError("C must be (d, r) and X (r, n)")
    rho0 = _uniform_diag(R0, d, "R")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)

    Epred = np.zeros([1, Iter + 1]); Efull = np.zeros([1, Iter + 1])
    Epred[:, 0] = Einit; Efull[:, 0] = Einit
    EfullSmooth = np.zeros([1, Iter + 1]); EfullSmooth[:, 0] = Einit
    RunTime = np.zeros([1, Iter + 1])
    t0 = time.time()

    # ingest on the device: (d, n) -> time-major (n, d), so that y_t / m_t are contiguous (the reference gathers a strided
    # column per step); M and Mmiss travel as one byte per entry
    Yt, _ = ingest(Y, dtype=dtype, keep_nan=False, want_mask=False, device=dev.index)
    Mt = transpose_mask(M, device=dev.index)
    Yo, _ = ingest(YorigInt, dtype=dtype, keep_nan=False, want_mask=False, device=dev.index)
    Et = transpose_mask(Mmiss, device=dev.index)

    rho_vector = np.ndim(rho0) != 0
    rho_arg = rho0 if rho_vector else [rho0]
    eng = FilterEngine(d, r, dtype=dtype, robust=robust, c_update_transpose=robust, dynamics=_capi.DYN_IDENTITY,
                       device=dev.index, rho_vector=rho_vector)
    InsideBars = 0.0                                                            # Iter = 0: the bounds stay zero
    details = {}
    try:
        eng.set_state(C_=C, V=V, P=P, x=np.ascontiguousarray(X[:, n - 1]), Q=Q0, rho=rho_arg, lam=[lambda0 if robust else 0.0])
        for i in range(Iter):
            if robust:
                eng.set_state(Q=Q0, rho=rho_arg, lam=[lambda0])                # rPSMF.py:77-79
            # x_bar of t = 0 wraps to X[:, n-1] (rPSMF.py:86): that is the engine's carried x.  The evaluation of the
            # one-step predictions (Epred, the 2-sigma coverage) is accumulated inside the filter pass.
            out = eng.run(Yt, Mt, k0=1, want_X=True, want_scal=return_details, want_Yrec=return_details, Yorig=Yo, E=Et, sig=sig,
                          want_moments=smooth)
            bad = eng.status()
            if smooth:
                EfullSmooth[:, i + 1] = _smoothed_efull(eng, out["moments"], Yo, Et)[0]
            ev = out["eval"].cpu().numpy().reshape(-1)
            ef = eng.eval_full(out["X"], Yo, Et).cpu().numpy().reshape(-1)      # (C X - Yorig)^2 over Mmiss, final C (rPSMF.py:137)
            X[:, :] = out["X"].cpu().numpy().T                                  # rPSMF.py:104 (in place)
            Epred[:, i + 1] = np.sqrt(ev[_capi.EVAL_SSE] / ev[_capi.EVAL_COUNT])   # common.py:79-84
            Efull[:, i + 1] = np.sqrt(ef[0] / ef[1])
            InsideBars = float(ev[_capi.EVAL_INSIDE] / ev[_capi.EVAL_COUNT])    # common.py:87-94 (bounds of the last sweep)
            if bad >= 0:
                Epred[:, i + 1] = np.nan; Efull[:, i + 1] = np.nan; EfullSmooth[:, i + 1] = np.nan
            RunTime[:, i + 1] = time.time() - t0
            if return_details:
                st = eng.get_state()
                details = dict(C=st["C"].to(torch.float64).cpu().numpy(), Yrec=out["Yrec"].to(torch.float64).cpu().numpy().T,
                               scal=out["scal"].cpu().numpy(), state=st, launch=eng.launch_info())
    finally:
        eng.close()
    res = (Epred, Efull, RunTime, InsideBars) + ((EfullSmooth,) if smooth else ())
    if return_details:
        return res + (details,)
    return res


def _smoothed_efull(eng, moments, Yo, Et):
    """Efull of the smoothed states, one value per series: sqrt of the mean of (C_T X^s - Yorig)^2 over Mmiss, NaN for a series
    whose smoothed states are not finite (the smoother met a singular P_bar); the other series keep their value."""
    Xs = eng.smooth(moments, check=False).reshape(eng.S, -1, eng.r)
    finite = torch.isfinite(Xs).reshape(eng.S, -1).all(dim=1).cpu().numpy()
    ef = eng.eval_full(Xs, Yo, Et).cpu().numpy().reshape(eng.S, 2)
    return np.where(finite, np.sqrt(ef[:, 0] / ef[:, 1]), np.nan)


def robust_PSMF(Y, C, X, d, n, r, M, Mmiss, V, Q0, R0, P, lambda0, sig, Iter, YorigInt, Einit, *, smooth=False):
    """ExperimentImpute/rPSMF.py:39-58 signature."""
    return _fit(Y, C, X, d, n, r, M, Mmiss, V, Q0, R0, P, lambda0, sig, Iter, YorigInt, Einit, robust=True, smooth=smooth)


def ProbabilisticSequentialMatrixFactorizer(Y, C, X, d, n, r, M, Mmiss, lam, V, Q, R, P, sig, Iter, YorgInt, Einit, *, smooth=False):
    """ExperimentImpute/PSMF.py:40-42 signature (``lam`` is unused there too)."""
    return _fit(Y, C, X, d, n, r, M, Mmiss, V, Q, R, P, 0.0, sig, Iter, YorgInt, Einit, robust=False, smooth=smooth)


def fit_repeats(Ys, Cs, Xs, Ms, Mmisses, V, Q0, R0, P, lambda0, sig, Iter, YorigInt, Einits, robust=True, device=None,
                dtype=torch.float64, *, smooth=False):
    """All repeats of the imputation experiment in ONE batch (the 100-repeat loop of ExperimentImpute/rPSMF.py:194-232 /
    PSMF.py:140-178): repeat k has its own random mask and initial C, X but the same data set, so the repeats are
    independent series of equal shape, filtered side by side in one launch: one CTA per repeat while its C fits the shared
    memory of a CTA (the resident batch kernel) or its residuals do (the direct-load kernel), and above that a
    thread-block cluster of up to 16 CTAs per repeat, so data sets of some hundred thousand rows run as one batch too.
    Arguments are lists over the repeats of what ``robust_PSMF`` / ``ProbabilisticSequentialMatrixFactorizer``
    take per call; returns the lists ``(Epred, Efull, RunTime, InsideBars)`` of what they return per call.  ``Xs[k]`` is
    overwritten in place like ``X`` there.  ``smooth=True`` appends the list ``EfullSmooth`` (see the module docstring)."""
    S = len(Ys)
    d, n = np.asarray(Ys[0]).shape
    r = np.asarray(Cs[0]).shape[1]
    rho0 = _uniform_diag(R0, d, "R")
    if np.ndim(rho0) != 0:
        raise NotImplementedError("fit_repeats runs as one batched engine: R must be rho * I (use the per-repeat functions)")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    t0 = time.time()
    Yt = torch.stack([ingest(Ys[k], dtype=dtype, keep_nan=False, want_mask=False, device=dev.index)[0] for k in range(S)])
    Mt = torch.stack([transpose_mask(Ms[k], device=dev.index) for k in range(S)])
    Et = torch.stack([transpose_mask(Mmisses[k], device=dev.index) for k in range(S)])
    Yo1, _ = ingest(YorigInt, dtype=dtype, keep_nan=False, want_mask=False, device=dev.index)
    Yo = Yo1.unsqueeze(0).expand(S, n, d).contiguous()
    eng = FilterEngine(d, r, n_series=S, dtype=dtype, robust=robust, c_update_transpose=robust, dynamics=_capi.DYN_IDENTITY,
                       device=dev.index)
    Epred = [np.zeros([1, Iter + 1]) for _ in range(S)]
    Efull = [np.zeros([1, Iter + 1]) for _ in range(S)]
    RunTime = [np.zeros([1, Iter + 1]) for _ in range(S)]
    Inside = [0.0] * S
    EfullSmooth = [np.zeros([1, Iter + 1]) for _ in range(S)]
    for k in range(S):
        Epred[k][:, 0] = Einits[k]; Efull[k][:, 0] = Einits[k]; EfullSmooth[k][:, 0] = Einits[k]
    try:
        eng.set_state(C_=np.stack([np.asarray(c, dtype=np.float64) for c in Cs]), V=V, P=P,
                      x=np.stack([np.ascontiguousarray(np.asarray(x)[:, n - 1]) for x in Xs]), Q=Q0, rho=[rho0],
                      lam=[lambda0 if robust else 0.0])
        for i in range(Iter):
            if robust:
                eng.set_state(Q=Q0, rho=[rho0], lam=[lambda0])                 # rPSMF.py:77-79
            out = eng.run(Yt, Mt, k0=1, want_X=True, Yorig=Yo, E=Et, sig=sig, want_moments=smooth)
            bad = eng.status()
            efs = _smoothed_efull(eng, out["moments"], Yo, Et) if smooth else None
            ev = out["eval"].cpu().numpy().reshape(S, -1)
            Xd = out["X"].reshape(S, n, r)
            ef = eng.eval_full(Xd, Yo, Et).cpu().numpy().reshape(S, 2)
            Xh = Xd.cpu().numpy()
            for k in range(S):
                Xs[k][:, :] = Xh[k].T
                Epred[k][:, i + 1] = np.sqrt(ev[k, _capi.EVAL_SSE] / ev[k, _capi.EVAL_COUNT])
                Efull[k][:, i + 1] = np.sqrt(ef[k, 0] / ef[k, 1])
                Inside[k] = float(ev[k, _capi.EVAL_INSIDE] / ev[k, _capi.EVAL_COUNT])
                if smooth:
                    EfullSmooth[k][:, i + 1] = efs[k]
                if bad >= 0 and not np.isfinite(Xh[k]).all():
                    Epred[k][:, i + 1] = np.nan; Efull[k][:, i + 1] = np.nan
                    if smooth:
                        EfullSmooth[k][:, i + 1] = np.nan
                RunTime[k][:, i + 1] = (time.time() - t0) / S                  # wall time of the batch, shared evenly
        info = eng.launch_info()
    finally:
        eng.close()
    fit_repeats.last_launch = info
    if smooth:
        return Epred, Efull, RunTime, Inside, EfullSmooth
    return Epred, Efull, RunTime, Inside
