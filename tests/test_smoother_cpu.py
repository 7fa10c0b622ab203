# -*- coding: utf-8 -*-
"""The float64 restatement of the moment record and the RTS smoother (tests/smoother_oracle.py) against the dense joint
posterior of the linear-Gaussian model that non-robust PSMF with V = 0 is."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import smoother_oracle as so  # noqa: E402
from oracle import psmf_oracle as po  # noqa: E402


def _model(r, d, T, dyn, missing, seed):
    rng = np.random.default_rng(seed)
    C = rng.standard_normal((d, r))
    rho = 0.3
    B = rng.standard_normal((r, r))
    Q = 0.05 * (B @ B.T / r + np.eye(r))
    if dyn == "linear":
        A = 0.9 * np.linalg.qr(rng.standard_normal((r, r)))[0]
        c = 0.1 * rng.standard_normal(r)
    else:
        A, c = np.eye(r), np.zeros(r)
    mu0 = rng.standard_normal(r)
    B0 = rng.standard_normal((r, r))
    P0 = B0 @ B0.T / r + 0.5 * np.eye(r)
    Y = rng.standard_normal((T, d))
    M = np.ones((T, d))
    if missing:
        M = (rng.random((T, d)) > 0.3).astype(float)
        M[T // 2] = 0.0                                   # a step with every row missing
        Y = Y * M
    return C, rho, Q, A, c, mu0, P0, Y, M


@pytest.mark.parametrize("r", [1, 3, 5])
@pytest.mark.parametrize("dyn", ["identity", "linear"])
@pytest.mark.parametrize("missing", [False, True])
def test_rts_equals_dense_posterior(r, dyn, missing):
    C, rho, Q, A, c, mu0, P0, Y, M = _model(r, 12, 9, dyn, missing, seed=r + 10 * missing)
    rec = so.kalman_record(C, rho, Q, A, c, mu0, P0, Y, M)
    Xs, Ps = so.rts(rec, r)
    Xd, Pd = so.dense_posterior(C, rho, Q, A, c, mu0, P0, Y, M)
    assert np.max(np.abs(Xs - Xd)) < 1e-10 * max(1.0, np.max(np.abs(Xd)))
    assert np.max(np.abs(Ps - Pd)) < 1e-10 * max(1.0, np.max(np.abs(Pd)))
    # the last smoothed state is the filtered one; the smoothed covariance never exceeds the filtered one
    _, _, _, xT, PT = so.unpack(rec[-1], r)
    assert np.array_equal(Xs[-1], xT) and np.array_equal(Ps[-1], PT)
    for t in range(len(rec)):
        assert np.min(np.linalg.eigvalsh(so.unpack(rec[t], r)[4] - Ps[t])) > -1e-12


@pytest.mark.parametrize("dyn", ["identity", "linear"])
def test_oracle_record_is_the_kalman_filter_when_V_is_zero(dyn):
    """record_run on the oracle's own step (PSMF, V = 0, every row observed: a = 0, C fixed) is the textbook filter."""
    r = 4
    C, rho, Q, A, c, mu0, P0, Y, M = _model(r, 10, 7, dyn, False, seed=3)
    cfg = po.OracleConfig(robust=False, dynamics=po.DYN_LINEAR if dyn == "linear" else po.DYN_IDENTITY,
                          lin_A=A if dyn == "linear" else None, lin_c=c if dyn == "linear" else None)
    st = po.OracleState(C.copy(), mu0.copy(), P0.copy(), np.zeros((r, r)), Q.copy(), rho, 0.0)
    st2, rec = so.record_run(st, cfg, Y)
    ref = so.kalman_record(C, rho, Q, A, c, mu0, P0, Y, M)
    assert np.max(np.abs(rec - ref)) < 1e-12 * max(1.0, np.max(np.abs(ref)))
    assert np.array_equal(st2.C, C)


def test_record_layout():
    r = 3
    xb, F, Pb, x, P = (np.arange(r) + 1.0, np.arange(9.0).reshape(3, 3), -np.arange(9.0).reshape(3, 3), np.arange(r) + 10.0,
                       np.arange(9.0).reshape(3, 3) + 100)
    rec = so.pack(xb, F, Pb, x, P)
    assert rec.size == so.nmom(r) == 2 * r + 3 * r * r
    for a, b in zip(so.unpack(rec, r), (xb, F, Pb, x, P)):
        assert np.array_equal(a, b)
    from rpsmf_b200 import _capi
    off = _capi.MOM_OFFSETS(r)
    assert _capi.NMOM(r) == so.nmom(r)
    assert np.array_equal(rec[off["F"]:off["F"] + 9].reshape(3, 3), F) and np.array_equal(rec[off["x"]:off["x"] + r], x)
    assert np.array_equal(rec[off["Pbar"]:off["Pbar"] + 9].reshape(3, 3), Pb) and np.array_equal(rec[off["P"]:].reshape(3, 3), P)
