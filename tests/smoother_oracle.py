# -*- coding: utf-8 -*-
"""Float64 restatement of the per-step moment record (include/psmf_b200.h psmf_set_moments) and of the fixed-interval
(Rauch-Tung-Striebel) smoother (psmf_smooth) on top of the oracle's step.

    record     per step [x_bar | F | P_bar | x | P]: what entered the update and what left it, F the Jacobian of the predict
    rts        x^s_{T-1} = x_{T-1}, P^s_{T-1} = P_{T-1};  J_t = P_t F_{t+1}' P_bar_{t+1}^-1,
               x^s_t = x_t + J_t (x^s_{t+1} - x_bar_{t+1}),  P^s_t = P_t + J_t (P^s_{t+1} - P_bar_{t+1}) J_t'

Non-robust PSMF with V = 0 is exactly a linear-Gaussian state-space model with observation noise rho I on the observed rows
(C stays fixed, a = 0, omega = 1, P = K); ``dense_posterior`` conditions one (T r)-dimensional Gaussian for that model and
tests/test_smoother_cpu.py checks the restatement against it.  It lives beside the tests so that the pinned oracle stays as it is.
"""
from __future__ import annotations

import numpy as np

from oracle import psmf_oracle as po


def nmom(r):
    return 2 * r + 3 * r * r


def pack(xbar, F, Pbar, x, P):
    return np.concatenate([xbar.reshape(-1), F.reshape(-1), Pbar.reshape(-1), x.reshape(-1), P.reshape(-1)])


def unpack(rec, r):
    rr = r * r
    return (rec[:r], rec[r:r + rr].reshape(r, r), rec[r + rr:r + 2 * rr].reshape(r, r), rec[r + 2 * rr:2 * r + 2 * rr],
            rec[2 * r + 2 * rr:].reshape(r, r))


def record_run(st, cfg, Y, M=None, k0=1, xbar_F=None):
    """(final state, record (T, NMOM), X (T, r)) along the oracle's trajectory.  ``xbar_F``: per-step list of (x_bar, F) for
    external dynamics."""
    T = Y.shape[0]
    r = st.x.shape[0]
    rec = np.zeros((T, nmom(r)))
    for t in range(T):
        xf = xbar_F[t] if xbar_F is not None else po.dynamics(cfg.dynamics, st.theta, st.x, k0 + t, cfg)
        Pbar = xf[1] @ st.P @ xf[1].T + st.Q
        st, _ = po.step(st, cfg, Y[t], None if M is None else M[t], k=k0 + t, xbar_F=xf)
        rec[t] = pack(xf[0], xf[1], Pbar, st.x, st.P)
    return st, rec


def rts(rec, r):
    """(Xs (T, r), Ps (T, r, r)) of one series' record (T, NMOM)."""
    T = rec.shape[0]
    Xs, Ps = np.zeros((T, r)), np.zeros((T, r, r))
    _, _, _, Xs[T - 1], Ps[T - 1] = unpack(rec[T - 1], r)
    for t in range(T - 2, -1, -1):
        _, _, _, x0, P0 = unpack(rec[t], r)
        xb1, F1, Pb1, _, _ = unpack(rec[t + 1], r)
        J = np.linalg.solve(Pb1.T, F1 @ P0.T).T
        Xs[t] = x0 + J @ (Xs[t + 1] - xb1)
        Ps[t] = P0 + J @ (Ps[t + 1] - Pb1) @ J.T
    return Xs, Ps


def kalman_record(C, rho, Q, A, c, mu0, P0, Y, M):
    """Moment record of the textbook Kalman filter of x_t = A x_{t-1} + c + N(0, Q), y_t = C x_t + N(0, rho I) on the observed
    rows, x_0 ~ N(mu0, P0): the filter PSMF runs when V = 0 (P = (I + P_bar G)^-1 P_bar, G = C_o' C_o / rho)."""
    T, r = Y.shape[0], C.shape[1]
    rec = np.zeros((T, nmom(r)))
    x, P = mu0.copy(), P0.copy()
    for t in range(T):
        xb = A @ x + c
        Pb = A @ P @ A.T + Q
        o = M[t] > 0
        Co = C[o]
        G = Co.T @ Co / rho
        b = Co.T @ (Y[t][o] - Co @ xb) / rho
        K = np.linalg.solve(np.eye(r) + Pb @ G, Pb)
        x, P = xb + K @ b, K
        rec[t] = pack(xb, A, Pb, x, P)
    return rec


def dense_posterior(C, rho, Q, A, c, mu0, P0, Y, M):
    """Mean (T, r) and covariance (T, r, r) of x_t | y_{1:T}, by conditioning the joint Gaussian of (x_0, ..., x_T) in
    information form and marginalising x_0."""
    T, r = Y.shape[0], C.shape[1]
    n = (T + 1) * r
    Jm, h = np.zeros((n, n)), np.zeros(n)
    P0i, Qi = np.linalg.inv(P0), np.linalg.inv(Q)
    Jm[:r, :r] += P0i
    h[:r] += P0i @ mu0
    for t in range(1, T + 1):
        i0, i1 = slice((t - 1) * r, t * r), slice(t * r, (t + 1) * r)
        # (x_t - A x_{t-1} - c)' Qi (x_t - A x_{t-1} - c)
        Jm[i1, i1] += Qi
        Jm[i0, i0] += A.T @ Qi @ A
        Jm[i1, i0] -= Qi @ A
        Jm[i0, i1] -= A.T @ Qi
        h[i1] += Qi @ c
        h[i0] -= A.T @ Qi @ c
        o = M[t - 1] > 0
        Co = C[o]
        Jm[i1, i1] += Co.T @ Co / rho
        h[i1] += Co.T @ Y[t - 1][o] / rho
    cov = np.linalg.inv(Jm)
    mean = cov @ h
    X = mean[r:].reshape(T, r)
    Ps = np.stack([cov[(t + 1) * r:(t + 2) * r, (t + 1) * r:(t + 2) * r] for t in range(T)])
    return X, Ps
