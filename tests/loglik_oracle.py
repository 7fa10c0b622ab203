# -*- coding: utf-8 -*-
"""Float64 restatement of the per-step log-likelihood record (include/psmf_b200.h PSMF_LOGLIK) on top of the oracle's step.

Per step k, over the n = n_obs observed rows, with the state entering the step:

    nll_k    the incremental negative log-likelihood that the kernels' gradients differentiate (oracle.dll_df): y_obs under
             N(C_o x_bar, N I) or, with ll_student, the t_lambda law with that scale; N = x_bar' V x_bar + eta
    log p_k  log p(y_obs | past) under S_obs = C_o Pbar C_o' + diag(rho_i + a), Gaussian or (robust) multivariate t with
             lambda degrees of freedom; simplified: S_obs = diag(rho_i + a)

This restatement takes the kernels' route (matrix-determinant lemma, Woodbury); tests/test_loglik_cpu.py checks it against
dense densities built from S_obs itself.  It lives beside the tests so that the pinned oracle stays as it is.
"""
from __future__ import annotations

import numpy as np
from scipy.special import gammaln

from oracle import psmf_oracle as po


def nll_value(n, N, q1, lam, ll_student):
    """nll_k from n_obs, N, q1 = sum_obs e^2 and lambda; N and q1 may be complex (complex-step derivative)."""
    if n == 0:
        return 0.0
    if not ll_student:
        return 0.5 * n * np.log(2.0 * np.pi * N) + q1 / (2.0 * N)
    return (gammaln(0.5 * lam) - gammaln(0.5 * (lam + n)) + 0.5 * n * np.log(lam * np.pi * N)
            + 0.5 * (lam + n) * np.log(1.0 + q1 / (lam * N)))


def nll_of_f(f, V, eta, C_o, y_o, lam, ll_student):
    """nll_k as a function of f = x_bar with eta and V held fixed (the convention of oracle.dll_df)."""
    N = f @ V @ f + eta
    e = y_o - C_o @ f
    return nll_value(y_o.shape[0], N, e @ e, lam, ll_student)


def logpred_value(n, logdet, d2, lam, robust):
    if n == 0:
        return 0.0
    if not robust:
        return -0.5 * (n * np.log(2.0 * np.pi) + logdet + d2)
    return (gammaln(0.5 * (lam + n)) - gammaln(0.5 * lam) - 0.5 * n * np.log(lam * np.pi) - 0.5 * logdet
            - 0.5 * (lam + n) * np.log1p(d2 / lam))


def pbar_of(st, cfg, F):
    return st.P if cfg.simplified else F @ st.P @ F.T + st.Q


def step_loglik(st, cfg, y, m, k, ll_student, xbar_F=None):
    """(new_state, out, nll_k, log p_k) of one oracle step; out gains "S_obs" pieces for the dense checks."""
    d = st.C.shape[0]
    m = np.ones(d) if m is None else np.asarray(m, dtype=np.float64)
    xbar, F = xbar_F if xbar_F is not None else po.dynamics(cfg.dynamics, st.theta, st.x, k, cfg)
    new, out = po.step(st, cfg, y, m, k=k, xbar_F=xbar_F)
    S = out["stats"]
    n, a, N, lam = S["nobs"], out["a"], out["N"], st.lam
    obs = m > 0
    rho_i = (np.full(d, float(st.rho)) if np.ndim(st.rho) == 0 else np.asarray(st.rho))[obs]
    e_o = out["e"][obs]
    w = 1.0 / (rho_i + a)
    Pbar = pbar_of(st, cfg, F)
    ldr = float(np.sum(np.log(rho_i + a)))
    d2 = float(np.sum(w * e_o * e_o))
    if not cfg.simplified and n > 0:
        Mx = np.eye(xbar.shape[0]) + Pbar @ S["G"]
        sign, ld = np.linalg.slogdet(Mx)
        assert sign > 0
        ldr += ld
        d2 -= float(S["b"] @ np.linalg.solve(Mx, Pbar @ S["b"]))
    nll = nll_value(n, N, S["q1"], lam, ll_student)
    lp = logpred_value(n, ldr, d2, lam, cfg.robust)
    out = dict(out, Pbar=Pbar, rho_obs=rho_i, obs=obs, y_obs=np.asarray(y, dtype=np.float64)[obs], C_o=st.C[obs],
               V_in=st.V, lam_in=lam)
    return new, out, float(nll), float(lp)


def run_loglik(st, cfg, Y, M, ll_student, k0=1, record=None):
    """Per-step (nll (T,), logpred (T,)) along the oracle's trajectory; the final state too."""
    T = Y.shape[0]
    nll, lp = np.zeros(T), np.zeros(T)
    for t in range(T):
        st, out, nll[t], lp[t] = step_loglik(st, cfg, Y[t], None if M is None else M[t], k0 + t, ll_student)
        if record is not None:
            record.append(out)
    return st, nll, lp
