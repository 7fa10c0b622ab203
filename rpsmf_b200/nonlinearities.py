# -*- coding: utf-8 -*-
"""Dynamics f_theta(x, t) of the predict half of the filter step.

The CUDA kernel evaluates two dynamics on the device (with closed-form Jacobians):

* identity  -- ``RandomWalk`` (pypsmf/psmf/nonlinearities.py:42-56) and the imputation scripts
* ``cos(2 pi theta t + x)`` -- the ``nonlinearity`` of the synthetic experiments
  (ExperimentSynthetic/synthetic_psmf.py:105-106)

Any other callable ``f(theta, x, t) -> (r, 1)`` is supported through the external path: the host
evaluates f and its Jacobian once per step and the kernel runs one step per launch (slow, general).
``classify`` recognises the two built-ins either by their tag or by probing the callable, so the
reference's own ``RandomWalk()`` / ``nonlinearity`` objects select the device path unchanged.

A callable that is affine in x, ``f(theta, x, t) = A(theta) x + c(theta)``, can be marked with ``affine(f)``: the
classes then run it as device linear dynamics (one launch per sweep) and learn theta from the gradient with respect to
A and c that the kernels accumulate.  Unmarked callables keep the external path.
"""

from __future__ import annotations

import numpy as np

from . import _capi


class RandomWalk:
    """f(x) = x; takes no parameters (same call signature as the reference class)."""

    dims = []
    rank = 0
    n_params = 0
    _psmf_dynamics = _capi.DYN_IDENTITY

    def __call__(self, theta, x, t):
        return x


def cos_phase(theta, x, t):
    """cos(2 pi theta t + x), evaluated with the same operation order as the reference expression."""
    return np.cos(2 * np.pi * theta * t + x)


cos_phase._psmf_dynamics = _capi.DYN_COS


def classify(nonlinearity, r):
    """Return the PSMF_DYN_* id of a callable."""
    kind = getattr(nonlinearity, "_psmf_dynamics", None)
    if kind is not None:
        return int(kind)
    rng = np.random.RandomState(12345)
    is_id, is_cos = True, True
    for t in (1, 7, 123):
        theta = rng.rand(r, 1)
        x = rng.randn(r, 1)
        try:
            out = np.asarray(nonlinearity(theta, x, t), dtype=np.float64).reshape(r, 1)
        except Exception:
            try:   # parameter-free callables are often called with an empty / dummy theta
                out = np.asarray(nonlinearity(np.zeros((1, 1)), x, t), dtype=np.float64).reshape(r, 1)
                is_cos = False
            except Exception:
                return _capi.DYN_EXTERNAL
        is_id = is_id and np.array_equal(out, x)
        is_cos = is_cos and np.allclose(out, np.cos(2 * np.pi * theta * t + x), rtol=0, atol=1e-15)
    if is_id:
        return _capi.DYN_IDENTITY
    if is_cos:
        return _capi.DYN_COS
    return _capi.DYN_EXTERNAL


def jacobian_x(nonlinearity, theta, x, t):
    """F = d f / d x at (theta, x, t) as an (r, r) matrix.  (The reference uses autograd, psmf.py:44,108-114.)

    Central differences are always computed; when the callable also accepts complex input and its
    complex-step derivative agrees with them (i.e. it is analytic there), the complex-step value -- exact to
    rounding -- is returned instead."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, 1)
    r = x.shape[0]
    Fd = np.zeros((r, r))
    for j in range(r):
        h = 1e-6 * max(1.0, abs(float(x[j, 0])))
        xp, xm = x.copy(), x.copy()
        xp[j, 0] += h
        xm[j, 0] -= h
        Fd[:, j] = (np.asarray(nonlinearity(theta, xp, t), dtype=np.float64).reshape(r)
                    - np.asarray(nonlinearity(theta, xm, t), dtype=np.float64).reshape(r)) / (2 * h)
    try:
        Fc = np.zeros((r, r))
        h = 1e-30
        for j in range(r):
            xc = x.astype(np.complex128)
            xc[j, 0] += 1j * h
            out = np.asarray(nonlinearity(theta, xc, t))
            if not np.iscomplexobj(out):
                return Fd
            Fc[:, j] = np.imag(out).reshape(r) / h
        if np.all(np.isfinite(Fc)) and np.max(np.abs(Fc - Fd)) <= 1e-5 * max(1.0, float(np.max(np.abs(Fd)))):
            return Fc
    except Exception:
        pass
    return Fd


def jacobian_theta(nonlinearity, theta, x, t):
    """J = d f / d theta at (theta, x, t) as an (r, p) matrix, p = theta.size (the reference differentiates the
    incremental likelihood with autograd, psmf.py:41,167-177; here d ell / d f comes from the kernel and the chain
    rule is closed with this Jacobian).  Complex-step when the callable is analytic, else central differences."""
    theta = np.asarray(theta, dtype=np.float64)
    shape = theta.shape
    th = theta.reshape(-1)
    p = th.size
    r = np.asarray(x).reshape(-1).size
    Jd = np.zeros((r, p))
    for j in range(p):
        h = 1e-6 * max(1.0, abs(float(th[j])))
        tp, tm = th.copy(), th.copy()
        tp[j] += h
        tm[j] -= h
        Jd[:, j] = (np.asarray(nonlinearity(tp.reshape(shape), x, t), dtype=np.float64).reshape(r)
                    - np.asarray(nonlinearity(tm.reshape(shape), x, t), dtype=np.float64).reshape(r)) / (2 * h)
    try:
        Jc = np.zeros((r, p))
        h = 1e-30
        for j in range(p):
            tc = th.astype(np.complex128)
            tc[j] += 1j * h
            out = np.asarray(nonlinearity(tc.reshape(shape), x, t))
            if not np.iscomplexobj(out):
                return Jd
            Jc[:, j] = np.imag(out).reshape(r) / h
        if np.all(np.isfinite(Jc)) and np.max(np.abs(Jc - Jd)) <= 1e-5 * max(1.0, float(np.max(np.abs(Jd)))):
            return Jc
    except Exception:
        pass
    return Jd


class affine:
    """Marks ``f(theta, x, t) = A(theta) x + c(theta)`` (affine in x, independent of t) for the device linear dynamics.
    Calls go to ``f`` unchanged; ``parts`` checks the claim at a given theta and extracts A and c."""

    _psmf_dynamics = _capi.DYN_LINEAR

    def __init__(self, f):
        self.f = f

    def __call__(self, theta, x, t):
        return self.f(theta, x, t)

    def _eval(self, theta, x, t, r):
        return np.asarray(self.f(theta, np.asarray(x, dtype=np.float64).reshape(r, 1), t), dtype=np.float64).reshape(r)

    def parts(self, theta, r):
        """(A (r, r), c (r)) at theta: A = [f(theta, e_j) - f(theta, 0)], c = f(theta, 0).  Raises ValueError when f is not
        affine in x or depends on t at this theta (checked on a few probes)."""
        eye = np.eye(r)
        c = self._eval(theta, np.zeros(r), 1, r)
        A = np.stack([self._eval(theta, eye[j], 1, r) - c for j in range(r)], axis=1)
        rng = np.random.RandomState(2024)
        for t in (1, 7, 123):
            x = rng.randn(r)
            want = A @ x + c
            got = self._eval(theta, x, t, r)
            scale = max(1.0, float(np.max(np.abs(A))) * float(np.max(np.abs(x))) + float(np.max(np.abs(c))))
            if not np.all(np.isfinite(got)) or np.max(np.abs(got - want)) > 1e-10 * scale:
                raise ValueError("affine(f): f(theta, x, t) is not A x + c at this theta (not affine in x, or it depends on t)")
        return A, c

    def theta_jacobians(self, theta, r):
        """(dA/dtheta (r, r, p), dc/dtheta (r, p)) at theta, from jacobian_theta at x = 0 and x = e_j."""
        eye = np.eye(r)
        J0 = jacobian_theta(self.f, theta, np.zeros((r, 1)), 1)
        dA = np.stack([jacobian_theta(self.f, theta, eye[j].reshape(r, 1), 1) - J0 for j in range(r)], axis=1)
        return dA, J0
