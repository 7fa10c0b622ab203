# -*- coding: utf-8 -*-
"""Class surface of pypsmf (pypsmf/psmf/psmf.py, rpsmf.py) on top of the CUDA filter engine.

    PSMFIter, PSMFRecursive                      pypsmf/psmf/psmf.py:14-248, 275-331
    rPSMFIter, rPSMFIterMissing, rPSMFRecursive  pypsmf/psmf/rpsmf.py:11-184, 187-287, 290-334

Same constructor signatures, same ``run`` / ``step`` / ``predict`` / ``optim_*`` methods, same post-fit
state dictionaries (``_C[T]``, ``_mu[T]``, ``_P[T]``, ``_V[T]``, ``_theta[i]``, ``_y_pred[k]``,
``_mu_pred[k]``, ``_lambda``, ``_Q``, ``_R``) and 1-based ``y = {k: (d, 1) ndarray}`` input.

What differs, by design:

* a whole sweep (``step``) is ONE kernel launch: the ten ``_hook`` methods of ``PSMFIter.inner``
  (psmf.py:90-165) are fused into the CUDA step and cannot be overridden from Python.  The variant used
  by the synthetic experiments (ExperimentSynthetic/synthetic_psmf.py:78-100: P_bar = P, eta = tr(R)/d,
  x_t = x_bar) is the constructor flag ``simplified=True``; ``step_reset`` may still be overridden.
* R must be rho * I and Q, R constant over k (true for every experiment of the reference); anything else
  raises ``NotImplementedError``.
* the theta gradient of the incremental likelihood is accumulated on the device in closed form for the
  built-in ``cos(2 pi theta t + x)`` dynamics (the reference differentiates with autograd).  A callable marked
  with ``nonlinearities.affine`` (f = A(theta) x + c(theta)) runs as device linear dynamics: A and c are extracted once
  per sweep (per ``update_every`` block in the Recursive variants), the kernel accumulates the gradient with respect to
  A and c, and the host closes the chain rule with dA/dtheta, dc/dtheta.  Other callables run through the
  one-launch-per-step external path, with the theta gradient from the host Jacobian of each step.
* ``rPSMFIterMissing`` is bound to the masked semantics of ExperimentImpute/rPSMF.py (R_bar = M R M +
  (x'Vx) I), because the class as shipped in the reference is singular for any missing entry
  (SURVEY.md 3.3).
* ``loglik=True`` (keyword-only, all classes): sweep i also records ``_objective[i]`` = sum_k nll_k, the summed incremental
  negative log-likelihood whose gradient the optimisers descend, and ``_logpred[i]`` = sum_k log p(y_k | y_<k), the
  one-step predictive log-likelihood, both computed in the filter kernel (include/psmf_b200.h PSMF_LOGLIK).  The Recursive
  variants make one sweep: key 1, summed over their ``update_every`` blocks.
"""

from __future__ import annotations

import numpy as np
import torch

from . import _capi
from .engine import FilterEngine
from .learning_rate import BaseLearningRate, ConstantLearningRate
from .nonlinearities import classify, jacobian_theta, jacobian_x

_HOOKS = ("inner", "_predictive_mean", "_predictive_covariance", "_predict_measurement", "_compute_eta_k",
          "_compute_dictionary_innovation", "_update_dictionary_mean", "_update_dictionary_covariance",
          "_compute_inverse_coefficient_innovation", "_update_coefficient_mean", "_update_coefficient_covariance",
          "_store_gradient")


def _uniform_rho(R, d, what):
    """diag(R): a float for R = rho * I, the (d,) vector for a non-uniform diagonal (psmf.py:144-152 takes the Woodbury
    branch for any diagonal R); a non-diagonal R (the reference's O(d^3) fallback, psmf.py:150-152) is rejected."""
    R = np.asarray(R, dtype=np.float64)
    if R.ndim == 0:
        return float(R)
    if R.shape != (d, d):
        raise ValueError("%s must be (d, d)" % what)
    dg = np.diagonal(R)
    if np.count_nonzero(R - np.diag(dg)):
        raise NotImplementedError("%s must be diagonal; see rpsmf_b200/psmf.py" % what)
    if np.all(dg == dg[0]):
        return float(dg[0])
    return np.ascontiguousarray(dg, dtype=np.float64)


def _constant_over_k(D, what):
    """Qs / Rs of PSMFIter are dicts {k: matrix}; the kernel needs them constant over k."""
    if not isinstance(D, dict):
        return np.asarray(D, dtype=np.float64)
    vals = list(D.values())
    first = vals[0]
    for v in vals[1:]:
        if v is not first and not np.array_equal(v, first):
            raise NotImplementedError("%s must not depend on k" % what)
    return np.asarray(first, dtype=np.float64)


class PSMFIter:
    """Iterative PSMF (pypsmf/psmf/psmf.py:14-248)."""

    _robust = False
    _masked = False
    _ll_student = False

    def __init__(self, theta0, C0, V0, mu0, P0, Qs, Rs, nonlinearity, optim="adam", simplified=False, device=None,
                 dtype=torch.float64, *, loglik=False):
        self.nonlinearity = nonlinearity
        assert optim in ["adam", "sgd"]
        self.optim = optim
        for klass in type(self).__mro__:
            if klass.__module__.startswith("rpsmf_b200"):
                break                                   # library classes do not define the hooks
            for name in _HOOKS:
                if name in klass.__dict__:
                    raise NotImplementedError(
                        "%s overrides %s(): the per-step hooks are fused into the CUDA kernel. Use simplified=True "
                        "for the ExperimentSynthetic variant." % (klass.__name__, name))
        self.theta0 = theta0
        self.C0 = C0
        self.V0 = V0
        self.mu0 = mu0
        self.P0 = P0
        self._d, self._r = C0.shape
        self._C = {}
        self._P = {}
        self._Q = Qs
        self._R = Rs
        self._V = {}
        self._mu = {}
        self._theta = {0: theta0}
        self._y_pred = {}
        self._simplified = bool(simplified)
        self._device = device
        self._dtype = dtype
        self._dyn = classify(nonlinearity, self._r)
        self._engine = None
        self._ycache = None
        self._alpha = 1.0
        self._beta = 1.0
        self._gradsum = np.zeros(np.asarray(theta0).shape)
        self._loglik = bool(loglik)
        self._objective = {}
        self._logpred = {}
        self._llsum = None

    # ---- configuration handed to the kernel ----------------------------------------------------------
    def _q_rho(self):
        Q = _constant_over_k(self._Q, "Q")
        rho = _uniform_rho(_constant_over_k(self._R, "R"), self._d, "R")
        return Q, rho

    def _lambda0_value(self):
        return 0.0

    def _get_engine(self):
        if self._engine is None:
            self._rho_vector = np.ndim(self._q_rho()[1]) != 0
            self._engine = FilterEngine(
                self._d, self._r, dtype=self._dtype, robust=self._robust, simplified=self._simplified,
                c_update_transpose=True, fixed_lambda=getattr(self, "fixed_lambda", False), ll_student=self._ll_student,
                dynamics=self._dyn, alpha=self._alpha, beta=self._beta, device=self._device, rho_vector=self._rho_vector,
                grad_linear=self._dyn == _capi.DYN_LINEAR, loglik=self._loglik)
        return self._engine

    def _device_y(self, y, T, m=None):
        key = (id(y), T, id(m))
        if self._ycache is None or self._ycache[0] != key:
            eng = self._get_engine()
            Y = np.stack([np.asarray(y[k], dtype=np.float64).reshape(self._d) for k in range(1, T + 1)])
            Yd = torch.as_tensor(Y, dtype=self._dtype).to(eng.device)
            Md = None
            if m is not None:
                Mh = np.stack([np.asarray(m[k]).reshape(self._d) != 0 for k in range(1, T + 1)]).astype(np.uint8)
                Md = torch.as_tensor(Mh).to(eng.device)
            self._ycache = (key, Yd, Md)
        return self._ycache[1], self._ycache[2]

    def _theta_vec(self, theta):
        th = np.zeros(self._r)
        t = np.asarray(theta, dtype=np.float64).reshape(-1)
        th[: min(self._r, t.size)] = t[: self._r]
        return th

    # ---- reference API -------------------------------------------------------------------------------
    def run(self, y, T, n_iter, n_pred):
        self.optim_init()
        for i in range(1, n_iter + 1):
            self.step(y, i, T)
            self.predict(i, T, n_pred)
            self.optim_update(i)

    def step_reset(self):
        latest = lambda D, init: D[sorted(D.keys())[-1]] if D else init
        self._C = {0: latest(self._C, self.C0)}
        self._mu = {0: latest(self._mu, self.mu0)}
        self._P = {0: latest(self._P, self.P0)}
        self._V = {0: latest(self._V, self.V0)}
        self._gradsum = np.zeros(np.asarray(self.theta0).shape)
        self._yrec_from = None

    def step(self, y, i, T):
        self.step_reset()
        self._loglik_begin()
        self._sweep(y, None, self._theta[i - 1], 1, T)
        self._loglik_store(i)

    def _loglik_begin(self):
        self._llsum = None

    def _add_loglik(self, out):
        if self._loglik:
            s = torch.stack([out["nll"].sum(), out["logpred"].sum()])       # on the device: no transfer per block
            self._llsum = s if self._llsum is None else self._llsum + s

    def _loglik_store(self, i):
        if self._loglik:
            self._objective[i], self._logpred[i] = (self._llsum.tolist() if self._llsum is not None else [0.0, 0.0])

    def _sweep(self, y, m, theta, k_first, k_last, materialize=True):
        """Filter steps k_first..k_last (1-based, inclusive) with a fixed theta; state dicts move from
        key k_first - 1 to key k_last.  ``materialize=False`` (inner blocks of the Recursive variants): the state and the
        predictions stay on the device -- only the status word and the r-dim theta-gradient cross PCIe -- and the host
        dicts are filled by the next materialising sweep, for all the steps filtered since the last one."""
        eng = self._get_engine()
        T_all = max(y.keys()) if isinstance(y, dict) else len(y)
        Yd, Md = self._device_y(y, T_all, m)
        k0 = k_first - 1
        if k0 == 0 or not getattr(self, "_state_on_device", False):
            Q, rho = self._q_rho()
            eng.set_state(C_=np.asarray(self._C[k0], dtype=np.float64), V=self._V[k0], P=self._P[k0],
                          x=np.asarray(self._mu[k0], dtype=np.float64).reshape(-1), Q=Q, rho=rho if np.ndim(rho) else [rho],
                          lam=[self._lambda_entering(k0)], theta=self._theta_vec(theta))
        else:
            eng.set_state(theta=self._theta_vec(theta))
        n = k_last - k_first + 1
        ysl = Yd[k_first - 1:k_last]
        msl = None if Md is None else Md[k_first - 1:k_last]
        # one-step predictions of the steps filtered since the last materialising sweep: (T, d) on the device
        buf = getattr(self, "_yrec_dev", None)
        if buf is None or buf.shape != Yd.shape or buf.device != Yd.device:
            buf = self._yrec_dev = torch.empty_like(Yd)
            self._yrec_from = k_first
        if getattr(self, "_yrec_from", None) is None:
            self._yrec_from = k_first
        if self._dyn == _capi.DYN_EXTERNAL:
            buf[k_first - 1:k_last] = self._sweep_external(eng, ysl, msl, theta, k_first, n)     # accumulates self._gradsum itself
            grad = None
        elif self._dyn == _capi.DYN_LINEAR:
            eng.set_linear_dynamics(*self.nonlinearity.parts(theta, self._r))
            learn = np.asarray(theta).size > 0
            out = eng.run(ysl, msl, k0=k_first, want_X=False, Yrec_out=buf[k_first - 1:k_last].unsqueeze(0), want_grad=learn,
                          want_loglik=self._loglik)
            self._add_loglik(out)
            grad = None
            if learn:
                # d ell / d theta_p = <dA/dtheta_p, G_A>_F + <dc/dtheta_p, G_c>
                dA, dc = self.nonlinearity.theta_jacobians(theta, self._r)
                g = np.einsum("ij,ijp->p", out["grad_A"].cpu().numpy(), dA) + out["grad_c"].cpu().numpy() @ dc
                self._gradsum = self._gradsum + g.reshape(self._gradsum.shape)
        else:
            out = eng.run(ysl, msl, k0=k_first, want_X=False, Yrec_out=buf[k_first - 1:k_last].unsqueeze(0),
                          want_grad=self._dyn == _capi.DYN_COS, want_loglik=self._loglik)
            self._add_loglik(out)
            grad = out.get("grad")
        bad = eng.status()
        if bad >= 0:
            raise FloatingPointError("non-finite filter state at step %d" % (k_first + bad))
        if grad is not None:
            g = grad.cpu().numpy().reshape(-1)
            gs = np.zeros(self._gradsum.size)
            gs[: min(gs.size, g.size)] = g[: gs.size]
            self._gradsum = self._gradsum + gs.reshape(self._gradsum.shape)
        self._state_on_device = True
        if not materialize:
            return
        k_from, self._yrec_from = self._yrec_from, None
        st = eng.get_state()
        Yh = buf[k_from - 1:k_last].to(torch.float64).cpu().numpy()
        if Md is not None:
            Yh = Yh * Md[k_from - 1:k_last].cpu().numpy()     # masked prediction, rpsmf.py:229-230
        for j in range(k_last - k_from + 1):
            self._y_pred[k_from + j] = Yh[j].reshape(self._d, 1)
        self._C = {k_last: st["C"].to(torch.float64).cpu().numpy()}
        self._mu = {k_last: st["x"].cpu().numpy().reshape(self._r, 1)}
        self._P = {k_last: st["P"].cpu().numpy()}
        self._V = {k_last: st["V"].cpu().numpy()}
        self._after_sweep(st, k_last)

    def _sweep_external(self, eng, ysl, msl, theta, k_first, n):
        """Arbitrary callable dynamics: x_bar and F = df/dx from the host, one step per launch."""
        Yrec = torch.empty((n, self._d), dtype=self._dtype, device=eng.device)
        learn = np.asarray(theta).size > 0
        for j in range(n):
            k = k_first + j
            x = eng.get_state(want_C=False)["x"].cpu().numpy().reshape(self._r, 1)
            xbar = np.asarray(self.nonlinearity(theta, x, k), dtype=np.float64).reshape(self._r)
            F = None if self._simplified else jacobian_x(self.nonlinearity, theta, x, k)
            out = eng.run(ysl[j:j + 1], None if msl is None else msl[j:j + 1], k0=k, want_X=False, Yrec_out=Yrec[j:j + 1],
                          xbar=xbar, F=F, want_grad=learn, want_loglik=self._loglik)
            self._add_loglik(out)
            if learn:
                # d ell_k / d theta = J_theta' d ell_k / d f  (psmf.py:167-177): the kernel returns d ell_k / d f
                gf = out["grad"].cpu().numpy().reshape(self._r)
                J = jacobian_theta(self.nonlinearity, theta, x, k)
                self._gradsum = self._gradsum + (J.T @ gf).reshape(self._gradsum.shape)
        return Yrec

    def _lambda_entering(self, k0):
        return 0.0

    def _after_sweep(self, st, k_last):
        pass

    def predict(self, i, T, n_pred):
        self._predict_with(self._theta[i - 1], T, n_pred)

    def _predict_with(self, theta, T, n_pred):
        """psmf.py:182-188 on the device: an r-dim roll-out of mu through f (one warp) and ONE d x r . r x n_pred product
        with the filtered dictionary -- no per-horizon-step GEMV, nothing but the (n_pred, d) result crosses PCIe."""
        self._mu_pred = {T: self._mu[T]}
        if n_pred <= 0:
            return
        eng = self._get_engine()
        if not getattr(self, "_state_on_device", False):
            Q, rho = self._q_rho()
            eng.set_state(C_=np.asarray(self._C[T], dtype=np.float64), V=self._V[T], P=self._P[T],
                          x=np.asarray(self._mu[T], dtype=np.float64).reshape(-1), Q=Q, rho=rho if np.ndim(rho) else [rho],
                          lam=[self._lambda_entering(T)])
        if self._dyn == _capi.DYN_EXTERNAL:
            # the callable lives on the host: roll mu out here (r values per step), project on the device
            mus, mu = [], self._mu[T]
            for k in range(T + 1, T + n_pred + 1):
                mu = np.asarray(self.nonlinearity(theta, mu, k), dtype=np.float64).reshape(self._r, 1)
                mus.append(mu.reshape(-1))
            Xo, Yp = eng.predict(n_pred, T + 1, Xpred=np.stack(mus))
        else:
            eng.set_state(theta=self._theta_vec(theta))
            if self._dyn == _capi.DYN_LINEAR:
                eng.set_linear_dynamics(*self.nonlinearity.parts(theta, self._r))
            Xo, Yp = eng.predict(n_pred, T + 1)
        Xh = Xo.cpu().numpy()
        Yh = Yp.to(torch.float64).cpu().numpy()
        for j, k in enumerate(range(T + 1, T + n_pred + 1)):
            self._mu_pred[k] = Xh[j].reshape(self._r, 1)
            self._y_pred[k] = Yh[j].reshape(self._d, 1)

    # ---- optimisers (psmf.py:190-248) ------------------------------------------------------------------
    def adam_init(self, gam=1e-3, b1=0.9, b2=0.999):
        self.adam_gam = gam if isinstance(gam, BaseLearningRate) else ConstantLearningRate(gam)
        self.adam_b1 = b1
        self.adam_b2 = b2
        shape = np.asarray(self.theta0).shape
        self.adam_m = np.zeros(shape)
        self.adam_v = np.zeros(shape)
        self.adam_m_hat = np.zeros(shape)
        self.adam_v_hat = np.zeros(shape)

    def sgd_init(self, gam=1e-3):
        self.sgd_gam = gam if isinstance(gam, BaseLearningRate) else ConstantLearningRate(gam)

    def optim_init(self, gam=1e-3):
        if self.optim == "adam":
            self.adam_init(gam=gam)
        elif self.optim == "sgd":
            self.sgd_init(gam=gam)

    def optim_update(self, i, project=True):
        if self.optim == "adam":
            return self.adam_update(i, project=project)
        elif self.optim == "sgd":
            return self.sgd_update(i, project=project)

    def adam_update(self, i, project=True):
        g = self._gradsum
        self.adam_m = self.adam_b1 * self.adam_m + (1 - self.adam_b1) * g
        self.adam_v = self.adam_b2 * self.adam_v + (1 - self.adam_b2) * np.multiply(g, g)
        self.adam_m_hat = self.adam_m / (1 - np.power(self.adam_b1, i))
        self.adam_v_hat = self.adam_v / (1 - np.power(self.adam_b2, i))
        pr = np.divide(np.ones(np.asarray(self.theta0).shape), np.sqrt(self.adam_v_hat) + 1e-8)
        lr = self.adam_gam.get(i)
        self._theta[i] = self._theta[i - 1] - lr * np.multiply(pr, self.adam_m_hat)
        if project:
            self._theta[i] = np.maximum(self._theta[i], 0)

    def sgd_update(self, i, project=True):
        lr = self.sgd_gam.get(i)
        self._theta[i] = self._theta[i - 1] - lr * self._gradsum
        if project:
            self._theta[i] = np.maximum(self._theta[i], 0)

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None


class PSMFIterMissing(PSMFIter):
    def __init__(*args, **kwargs):
        # psmf.py:251-254: "WORK IN PROGRESS, DO NOT USE" in the reference as well
        raise NotImplementedError


class _RecursiveMixin:
    """theta is updated every `update_every` steps inside the sweep (psmf.py:275-331, rpsmf.py:290-334)."""

    def run(self, y, T, n_pred, update_every=1):
        self._update_every = update_every
        self.optim_init()
        self.step(y, T)
        self.predict(T, n_pred)

    def step(self, y, T):
        self.step_reset()
        self._loglik_begin()
        k = 1
        ue = max(1, int(self._update_every))
        while k <= T:
            k_last = min(T, ((k - 1) // ue + 1) * ue)
            # state and predictions stay on the device between the blocks; the dicts are filled once, after step T
            self._sweep(y, None, self._theta[k - 1], k, k_last, materialize=(k_last == T))
            for kk in range(k, k_last):
                self._carry_theta(kk)
            if k_last % ue == 0:
                self.optim_update(k_last)
                self._reset_gradient()
            else:
                self._carry_theta(k_last)
            k = k_last + 1
        self._loglik_store(1)

    def _reset_gradient(self):
        self._gradsum = np.zeros(np.asarray(self.theta0).shape)

    def _carry_theta(self, i):
        self._theta[i] = self._theta[i - 1]

    def predict(self, T, n_pred):
        self._predict_with(self._theta[T], T, n_pred)


class PSMFRecursive(_RecursiveMixin, PSMFIter):
    pass

