# -*- coding: utf-8 -*-
"""The float64 restatement of the per-step log-likelihood record (tests/loglik_oracle.py), without a GPU.

* log p_k against a dense scipy multivariate_normal / multivariate_t log-density of y_obs with S_obs = C_o Pbar C_o' +
  diag(rho_i + a) built explicitly (diag(rho_i + a) alone when simplified): independent of the determinant lemma and of
  Woodbury, the route the kernels take.
* the complex-step derivative of nll_k with respect to f = x_bar against oracle.dll_df with n = n_obs: the value is the
  function whose gradient the kernels already return.
* a step with every row missing contributes 0 to both."""
import numpy as np
import pytest
from scipy.stats import multivariate_normal, multivariate_t

from oracle import psmf_oracle as po
from loglik_oracle import nll_of_f, run_loglik
from synth import impute_init, make_problem

T = 6


def _setup(d, r, robust, simplified, rho_vector, seed, masked=True):
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, missing=0.3 if masked else 0.0)
    init = impute_init(r)
    rho = 10.0 * (0.5 + np.random.RandomState(seed).rand(d)) if rho_vector else init["rho"]
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), rho, init["lam"])
    cfg = po.OracleConfig(robust=robust, simplified=simplified, c_update_transpose=True)
    return Y, M, st, cfg


CASES = [(robust, simp, rv) for robust in (False, True) for simp in (False, True) for rv in (False, True)]


@pytest.mark.parametrize("robust,simplified,rho_vector", CASES,
                         ids=["%s-%s-%s" % ("rpsmf" if a else "psmf", "simp" if b else "full", "rhovec" if c else "rho")
                              for a, b, c in CASES])
@pytest.mark.parametrize("r", [1, 3, 5])
def test_logpred_against_dense_density(r, robust, simplified, rho_vector):
    d = 11
    Y, M, st, cfg = _setup(d, r, robust, simplified, rho_vector, seed=40 + r)
    rec = []
    _, _, lp = run_loglik(st, cfg, Y, M, ll_student=robust, record=rec)
    for t, out in enumerate(rec):
        C_o, y_o = out["C_o"], out["y_obs"]
        S = np.diag(out["rho_obs"] + out["a"])
        if not simplified:
            S = S + C_o @ out["Pbar"] @ C_o.T
        mean = C_o @ out["xbar"]
        if robust:
            dense = multivariate_t(loc=mean, shape=S, df=out["lam_in"]).logpdf(y_o)
        else:
            dense = multivariate_normal(mean=mean, cov=S).logpdf(y_o)
        assert abs(lp[t] - dense) <= 1e-10 * abs(dense), (t, lp[t], dense)


@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r", [1, 4])
def test_nll_complex_step_is_dll_df(r, ll_student):
    d = 13
    Y, M, st, cfg = _setup(d, r, True, False, False, seed=60 + r)
    rec = []
    run_loglik(st, cfg, Y, M, ll_student=ll_student, record=rec)
    h = 1e-30
    for out in rec:
        f, V, eta, lam = out["xbar"], out["V_in"], out["eta"], out["lam_in"]
        C_o, y_o = out["C_o"], out["y_obs"]
        e = y_o - C_o @ f
        ref = po.dll_df(ll_student, f, V, C_o.T @ e, float(e @ e), eta, lam, float(y_o.shape[0]))
        cs = np.array([np.imag(nll_of_f(f + 1j * h * np.eye(r)[j], V, eta, C_o, y_o, lam, ll_student)) / h for j in range(r)])
        assert np.max(np.abs(cs - ref)) <= 1e-12 * np.max(np.abs(ref))


@pytest.mark.parametrize("robust", [False, True])
def test_all_missing_step_is_zero(robust):
    d, r = 9, 3
    Y, M, st, cfg = _setup(d, r, robust, False, False, seed=80)
    M[2] = 0
    Y = Y * M
    _, nll, lp = run_loglik(st, cfg, Y, M, ll_student=robust)
    assert nll[2] == 0.0 and lp[2] == 0.0
    assert np.all(nll[:2] != 0.0) and np.all(np.isfinite(lp[:2]))
