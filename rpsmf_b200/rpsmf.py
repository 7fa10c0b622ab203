# -*- coding: utf-8 -*-
"""Robust (Student-t) variants: rPSMFIter, rPSMFIterMissing, rPSMFRecursive (pypsmf/psmf/rpsmf.py)."""

from __future__ import annotations

from collections import defaultdict

import numpy as np
import torch

from .psmf import PSMFIter, _RecursiveMixin, _uniform_rho


class rPSMFIter(PSMFIter):
    """pypsmf/psmf/rpsmf.py:11-184.  omega_k / phi_k rescale P, Q, R and V; lambda grows by d per step."""

    _robust = True
    _ll_student = True

    def __init__(self, theta0, C0, V0, mu0, P0, Q0, R0, lambda0, nonlinearity, fixed_lambda=False, use_scaling=False,
                 optim="adam", simplified=False, device=None, dtype=torch.float64, *, loglik=False):
        assert optim in ["adam", "sgd"]
        super().__init__(theta0, C0, V0, mu0, P0, Q0, R0, nonlinearity, optim=optim, simplified=simplified,
                         device=device, dtype=dtype, loglik=loglik)
        self.Q0 = Q0
        self.R0 = R0
        self.lambda0 = lambda0
        self.fixed_lambda = fixed_lambda
        if fixed_lambda:
            self._lambda = defaultdict(lambda: lambda0)
        else:
            self._lambda = {0: lambda0}
        self._Q = {0: Q0}
        self._R = {0: R0}
        self._alpha = 1.0
        self._beta = 1.0
        if use_scaling:
            self._alpha = self.compute_scaling_factor(self._r * self._d, self._d)
            self._beta = self.compute_scaling_factor(self._r, self._d)

    def compute_scaling_factor(self, dim, offset, verbose=False):
        """KL-optimal covariance scale between two multivariate-t laws (rpsmf.py:75-104): the alpha that
        minimises KL( t_{lambda+offset}(0, I) || t_lambda(0, alpha I) ) in `dim` dimensions.  A one-off host
        scalar, evaluated with mpmath like the reference (high dimension defeats double precision)."""
        import mpmath as mp

        m = mp.mpf(dim)
        lmd = mp.mpf(self.lambda0)
        off = mp.mpf(offset)

        def integrand(v, alpha):
            return (mp.power(v / (1 + v), m / 2) / (v * mp.power(1 + v, (lmd + off) / 2.0))
                    * mp.log(1 + (lmd + off) / (alpha * lmd) * v))

        def objective(alpha):
            h2 = mp.beta(m / 2, (lmd + off) / 2) * mp.log(alpha)
            h3 = (1 + lmd / m) * mp.quad(lambda v: integrand(v, alpha), [0, mp.inf])
            return h2 + h3

        return float(mp.findroot(lambda alpha: mp.diff(objective, alpha), mp.mpf(1.0), verbose=verbose))

    def step_reset(self):
        super().step_reset()
        if self.fixed_lambda:
            self._lambda = defaultdict(lambda: self.lambda0)
        else:
            self._lambda = {0: self.lambda0}
        self._R = {0: self.R0}
        self._Q = {0: self.Q0}

    def _q_rho(self):
        return np.asarray(self.Q0, dtype=np.float64), _uniform_rho(self.R0, self._d, "R0")

    def _lambda_entering(self, k0):
        return float(self.lambda0)

    def _after_sweep(self, st, k_last):
        self._Q = {k_last: st["Q"].cpu().numpy()}
        # R = rho * I (or diag(rho_i)): materialised only for small d (the reference keeps a (d, d) array per step)
        if st["rho"].numel() > 1:
            rv = st["rho"].cpu().numpy()
            self._R = {k_last: np.diag(rv) if self._d <= 4096 else rv}
        else:
            rho = float(st["rho"])
            self._R = {k_last: rho * np.eye(self._d) if self._d <= 4096 else rho}
        if not self.fixed_lambda:
            self._lambda = {k_last: float(st["lam"])}


class rPSMFIterMissing(rPSMFIter):
    """Masked robust PSMF.  ``m = {k: (d, 1)}`` with 1 = observed; y must be zero where missing.
    Semantics of ExperimentImpute/rPSMF.py:81-135 (see the module docstring of rpsmf_b200.psmf)."""

    _masked = True
    _ll_student = False      # masked incremental likelihood is the Gaussian form (rpsmf.py:196-200)

    def run(self, y, T, n_iter, n_pred, m=None):
        if m is None:
            raise TypeError("rPSMFIterMissing.run needs the mask dict m = {k: (d, 1)}")
        self.optim_init()
        for i in range(1, n_iter + 1):
            self.step(y, m, i, T)
            self.predict(i, T, n_pred)
            self.optim_update(i)

    def step(self, y, m, i, T):
        self.step_reset()
        self._loglik_begin()
        self._sweep(y, m, self._theta[i - 1], 1, T)
        self._loglik_store(i)


class rPSMFRecursive(_RecursiveMixin, rPSMFIter):
    pass
