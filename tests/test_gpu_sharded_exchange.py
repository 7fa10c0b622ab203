# -*- coding: utf-8 -*-
"""Row sharding with the caller-driven statistics exchange (PSMF_XCHG_EXTERNAL), every shard held in one process.

An engine created with exchange="external", world_size=N, rank=i and d_global=d filters rows [b_i, e_i) of one series and
never touches a mailbox: psmf_run does the pass and leaves the statistics of its rows in the buffer of stats_buffer(), the
caller all-reduces that buffer, and psmf_run_finish does the r x r update and the rank-1 update of C.  So N such engines
can live on one GPU: run phase 1 on each, sum the buffers on the device in rank order starting from 0.0 (the order of
gather_ranks in psmf_filter.cuh, so the sum is the one the in-kernel exchange forms), copy the sum back, run phase 2 on each.
That covers all of the sharded arithmetic -- d_global in eta, omega, phi and lambda, per-shard tiles and grid reductions,
shards smaller than a tile, shards with no observed row -- without the transport; tests/multi_gpu_external_check.py ties
this emulation to the NVLink mailboxes once.

Every cell checks the whole series against the float64 oracle (fp64 1e-9, fp32 storage 1e-4 on fp32-rounded Y and C0),
that the replicated quantities are bit-identical on all ranks, that never-observed rows keep C bit for bit, and that every
rank ran the direct-load kernel.
"""

import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _compare, _engine_run, _oracle_run, _padded, _torch
from test_gpu_kernel_matrix import FLAG_CASES, SPLIT_RANKS, TOL32, _grad_reference, _rounded, _theta
from test_gpu_linear_grad import _dynamics, _linear_grad_reference
from test_gpu_loglik import _reference as _loglik_reference

pytestmark = pytest.mark.gpu

T = 12
RANKS = list(range(1, 17))
REPLICATED = ("x", "P", "V", "Q", "rho", "lam", "theta")


def _shard_rows(d, world):
    from rpsmf_b200 import shard_rows
    return [shard_rows(d, world, i) for i in range(world)]


# layout -> (d, row ranges, forced ctas per shard (0 = automatic), rows never observed)
LAYOUTS = {
    # 126 tiles; the last shard holds 41 tiles, its last one a single row (d % 32 == 1)
    "rows4001x3": (4001, _shard_rows(4001, 3), (0, 0, 0), ()),
    # a 1-row shard, a shard under one tile and boundaries inside tiles: shard_rows never cuts so, a multi-node caller may
    "uneven1000": (1000, [(0, 1), (1, 32), (32, 65), (65, 1000)], (0, 0, 0, 0), ()),
    # 32 rows and 1 row
    "rows33x2": (33, _shard_rows(33, 2), (0, 0), ()),
    # 42 tiles per shard: 3 CTAs (every CTA reads all partials) and 20 CTAs (the transposed reduce-scatter, cps > 16)
    "rows4001x3_ctas": (4001, _shard_rows(4001, 3), (3, 20, 0), ()),
    # the uneven split plus a fifth shard whose rows are never observed; 3 CTAs on the 935-row shard
    "uneven1100x5": (1100, [(0, 1), (1, 32), (32, 65), (65, 1000), (1000, 1100)], (0, 0, 0, 3, 0), tuple(range(1000, 1100))),
    # 9 tiles over 8 ranks: one tile each, the last shard 37 rows
    "rows261x8": (261, _shard_rows(261, 8), (0,) * 8, ()),
}


def _problem(layout, r, seed, missing=0.2, dead_rows=True):
    """Y, M, C0, x0 over the whole series and the rows that are never observed (two rows and the layout's own)."""
    d, _, _, never = LAYOUTS[layout]
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, missing=missing)
    dead = sorted(set(([1, d // 2] if dead_rows else []) + list(never)))
    if dead:
        M[:, dead] = 0
        Y = Y * M
    return Y, M, C0, x0, np.array(dead, dtype=int)


def _sharded_run(splits, r, Y, M, C0, x0, init, dtype=None, ctas=None, robust=True, theta=None, A=None, c=None,
                 want_grad=False, loglik=False, xbar_fn=None, steps=None, **kw):
    """Filter Y (T, d) with one external-exchange engine per row range of `splits`, one step per launch pair: phase 1 on
    every rank, the statistics buffers summed on the device in rank order from 0.0 and copied back, phase 2 on every rank.
    M None with nan_mask=True: Y carries NaN where missing.  `xbar_fn(x)` -> (xbar, F) drives external dynamics from the
    replicated x of rank 0.  Returns a dict of per-rank lists: X (T, r), Yrec (T, d_i), scal (T, 8 or 10), grad (T, ...)
    per step, state (get_state), info (launch_info), status (per step), and the engines' tensors Yd / Md."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    dtype = dtype or torch.float64
    N, Tn = len(splits), Y.shape[0]
    d = splits[-1][1]
    ctas = ctas or (0,) * N
    engs = []
    for i, (b, e) in enumerate(splits):
        eng = FilterEngine(e - b, r, dtype=dtype, robust=robust, kernel=1, exchange="external", world_size=N, rank=i, d_global=d,
                           ctas=ctas[i], loglik=loglik, **kw)
        eng.set_state(C_=C0[b:e], V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]], theta=theta)
        if A is not None:
            eng.set_linear_dynamics(A, c)
        engs.append(eng)
    dev = engs[0].device
    Yd = [_padded(np.ascontiguousarray(Y[None, :, b:e]), dtype, dev)[0][0] for b, e in splits]
    Md = [None if M is None else torch.as_tensor(np.ascontiguousarray(M[:, b:e])).to(dev) for b, e in splits]
    nsc = 10 if loglik else 8
    X = [torch.full((Tn, r), float("nan"), dtype=torch.float64, device=dev) for _ in range(N)]
    Yr = [torch.full((Tn, e - b), float("nan"), dtype=dtype, device=dev) for b, e in splits]
    Sc = [torch.full((Tn, nsc), float("nan"), dtype=torch.float64, device=dev) for _ in range(N)]
    bufs = [eng.stats_buffer() for eng in engs]
    grads = [[] for _ in range(N)]
    status = np.full((steps or Tn, N), -2)
    for t in range(steps or Tn):
        dyn = {}
        if xbar_fn is not None:
            xbar, F = xbar_fn(engs[0].get_state(want_C=False)["x"].cpu().numpy())
            dyn = dict(xbar=xbar, F=F)
        for i, eng in enumerate(engs):
            eng.run(Yd[i][t:t + 1], None if Md[i] is None else Md[i][t:t + 1], k0=1 + t, want_X=False, Yrec_out=Yr[i][t:t + 1], **dyn)
        tot = torch.zeros_like(bufs[0])
        for buf in bufs:
            tot += buf
        for buf in bufs:
            buf.copy_(tot)
        for i, eng in enumerate(engs):
            out = eng.run(Yd[i][t:t + 1], None if Md[i] is None else Md[i][t:t + 1], k0=1 + t, X_out=X[i][t:t + 1],
                          scal_out=Sc[i][t:t + 1], want_grad=want_grad, _finish=True, **dyn)
            if want_grad:
                g = [out["grad_A"].reshape(-1), out["grad_c"]] if "grad_A" in out else [out["grad"]]
                grads[i].append(torch.cat(g))
        for i, eng in enumerate(engs):
            status[t, i] = eng.status()
    res = dict(X=[x.cpu().numpy() for x in X], Yrec=[y.double().cpu().numpy() for y in Yr], scal=[s.cpu().numpy() for s in Sc],
               grad=[np.stack([g.cpu().numpy() for g in gs]) if gs else None for gs in grads],
               state=[{k: (v.double().cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()} for eng in engs],
               info=[eng.launch_info() for eng in engs], status=status, Yd=Yd, Md=Md, engines=engs)
    return res


def _close(res):
    for eng in res.pop("engines"):
        eng.close()


def _whole(res):
    """The sharded run in the form of test_gpu_filter._engine_run: rank 0's replicated outputs, Yrec and C concatenated."""
    st = dict(res["state"][0])
    st["C"] = np.concatenate([s["C"] for s in res["state"]])
    return res["X"][0], np.concatenate(res["Yrec"], axis=1), res["scal"][0], st, res["info"][0]


def _check_ranks(res, dead=(), C0=None, tag="f64"):
    """Replicated quantities bit-identical on every rank, never-observed rows keep C, the direct-load kernel everywhere,
    no bad step."""
    N = len(res["X"])
    assert (res["status"] == -1).all(), res["status"]
    for i in range(N):
        assert res["info"][i]["kernel"] == "direct", (i, res["info"][i])
        assert np.array_equal(res["X"][i], res["X"][0]), i
        assert np.array_equal(res["scal"][i], res["scal"][0]), i
        for k in REPLICATED:
            assert np.array_equal(res["state"][i][k], res["state"][0][k]), (i, k)
        if res["grad"][0] is not None:
            assert np.array_equal(res["grad"][i], res["grad"][0]), i
    if len(dead):
        C = _whole(res)[3]["C"]
        assert np.array_equal(C[dead], _rounded(C0, tag)[dead])


def _dtype(tag):
    torch = _torch()
    return (torch.float64, TOL) if tag == "f64" else (torch.float32, TOL32)


def _oracle(Y, M, C0, x0, init, cfg, tag):
    return _oracle_run(_rounded(Y, tag), M, _rounded(C0, tag), x0, init, cfg)


# ---- 1. every rank and storage type on two layouts ---------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["rows4001x3", "uneven1000"])
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", RANKS, ids=lambda r: "r%d" % r)
def test_rank_matrix_sharded(r, tag, layout):
    dtype, tol = _dtype(tag)
    d, splits, ctas, _ = LAYOUTS[layout]
    Y, M, C0, x0, dead = _problem(layout, r, seed=2000 + 17 * r + d % 89)
    init = impute_init(r)
    res = _sharded_run(splits, r, Y, M, C0, x0, init, dtype=dtype, ctas=ctas)
    _check_ranks(res, dead, C0, tag)
    _compare(_whole(res), _oracle(Y, M, C0, x0, init, po.OracleConfig(robust=True), tag), tol)
    _close(res)


# ---- 2. world sizes ------------------------------------------------------------------------------------------------------
WORLD_LAYOUTS = ["rows33x2", "rows4001x3_ctas", "uneven1000", "uneven1100x5", "rows261x8"]


@pytest.mark.parametrize("layout", WORLD_LAYOUTS)
@pytest.mark.parametrize("r", [1, 9, 16], ids=lambda r: "r%d" % r)
def test_world_sizes(r, layout):
    d, splits, ctas, _ = LAYOUTS[layout]
    Y, M, C0, x0, dead = _problem(layout, r, seed=2100 + r + d)
    init = impute_init(r)
    res = _sharded_run(splits, r, Y, M, C0, x0, init, ctas=ctas)
    _check_ranks(res, dead, C0)
    for i, c in enumerate(ctas):
        if c:
            assert res["info"][i]["ctas"] == c, (i, res["info"][i])
    _compare(_whole(res), _oracle(Y, M, C0, x0, init, po.OracleConfig(robust=True), "f64"), TOL)
    _close(res)


@pytest.mark.parametrize("layout", ["uneven1000", "rows4001x3_ctas", "rows261x8"])
@pytest.mark.parametrize("r", [1, 16], ids=lambda r: "r%d" % r)
def test_step_with_every_row_missing(r, layout):
    """Step 6 has no observed row on any shard: a pure prediction step (q0 / eta := 0, where the reference evaluates
    0 * inf), finite, x unchanged under identity dynamics, bit-identical on all ranks and within 1e-11 of one engine
    filtering the whole series with the fused direct-load kernel."""
    d, splits, ctas, _ = LAYOUTS[layout]
    Y, M, C0, x0, dead = _problem(layout, r, seed=2200 + r)
    M[6] = 0
    Y = Y * M
    init = impute_init(r)
    res = _sharded_run(splits, r, Y, M, C0, x0, init, ctas=ctas)
    _check_ranks(res, dead, C0)
    X, Yrec, scal, st, _ = _whole(res)
    assert np.isfinite(X).all() and np.isfinite(Yrec).all() and np.isfinite(scal).all()
    assert all(np.isfinite(v).all() for v in st.values() if v is not None)
    assert np.array_equal(X[6], X[5])
    one = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=1)
    assert one[4]["kernel"] == "direct"
    assert relerr(X, one[0]) < 1e-11 and relerr(st["C"], one[3]["C"]) < 1e-11 and relerr(Yrec, one[1]) < 1e-11
    for k in ("P", "V", "rho", "lam"):
        assert relerr(st[k], one[3][k]) < 1e-11, k
    _close(res)


# ---- 3. flags on the uneven 4-way split ------------------------------------------------------------------------------------
FLAG_RT = [(r, "f64") for r in SPLIT_RANKS] + [(9, "f32")]
FLAG_IDS = ["r%d-%s" % p for p in FLAG_RT]
UNEVEN = LAYOUTS["uneven1000"][1]
D_UNEVEN = 1000


@pytest.mark.parametrize("case", list(FLAG_CASES))
@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_flags_sharded(r, tag, case):
    from rpsmf_b200 import _capi
    ekw, okw, cos = FLAG_CASES[case]
    dtype, tol = _dtype(tag)
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=2300 + r)
    init = impute_init(r)
    ekw = dict(ekw)
    robust = ekw.pop("robust")
    theta = None
    if cos:
        theta = _theta(r)
        init["theta"] = theta
        ekw["dynamics"] = _capi.DYN_COS
        okw = dict(okw, dynamics=po.DYN_COS)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, robust=robust, theta=theta, **ekw)
    _check_ranks(res, dead, C0, tag)
    _compare(_whole(res), _oracle(Y, M, C0, x0, init, po.OracleConfig(**okw), tag), tol)
    _close(res)


@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_nan_mask_sharded_bit_identical(r, tag):
    dtype, _ = _dtype(tag)
    Y, M, C0, x0, _ = _problem("uneven1000", r, seed=2400 + r)
    init = impute_init(r)
    a = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype)
    Yn = np.where(M == 0, np.nan, Y)
    b = _sharded_run(UNEVEN, r, Yn, None, C0, x0, init, dtype=dtype, nan_mask=True)
    _check_ranks(a)
    _check_ranks(b)
    for k in ("X", "Yrec", "scal"):
        for i in range(len(UNEVEN)):
            assert np.array_equal(a[k][i], b[k][i]), (k, i)
    for i in range(len(UNEVEN)):
        for k in ("C",) + REPLICATED:
            assert np.array_equal(a["state"][i][k], b["state"][i][k]), (i, k)
    _close(a)
    _close(b)


@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_theta_gradient_sharded_unmasked(r, tag, ll_student):
    """Cos dynamics, no missing entry: the theta gradient of each one-step launch, summed by the caller, against the
    oracle's closed form (theta_grad_cos) step by step."""
    from rpsmf_b200 import _capi
    dtype, tol = _dtype(tag)
    Y, _, C0, x0 = make_problem(D_UNEVEN, r, T, seed=2500 + r, missing=0.0)
    init = impute_init(r)
    theta = _theta(r)
    init["theta"] = theta
    res = _sharded_run(UNEVEN, r, Y, None, C0, x0, init, dtype=dtype, theta=theta, want_grad=True, dynamics=_capi.DYN_COS,
                       ll_student=ll_student)
    _check_ranks(res)
    _compare(_whole(res), _oracle(Y, None, C0, x0, init, po.OracleConfig(robust=True, dynamics=po.DYN_COS), tag), tol)
    ref = _grad_reference(_rounded(Y, tag), None, _rounded(C0, tag), x0, init, ll_student, D_UNEVEN)
    assert relerr(res["grad"][0].sum(axis=0), ref) < tol
    _close(res)


@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_theta_gradient_sharded_masked(r, tag, ll_student):
    """Cos dynamics with missing entries: the summed gradient within 1e-11 of one engine filtering the whole series with
    the fused direct-load kernel, and against the masked restatement.  fp32 storage: the fused pass takes the next step's
    statistics from the updated row before it is rounded to float, the split path from the stored float, so there the
    bound is the fp32 tolerance."""
    from rpsmf_b200 import _capi
    dtype, tol = _dtype(tag)
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=2600 + r)
    init = impute_init(r)
    theta = _theta(r)
    init["theta"] = theta
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, theta=theta, want_grad=True, dynamics=_capi.DYN_COS,
                       ll_student=ll_student)
    _check_ranks(res, dead, C0, tag)
    one = _engine_run(D_UNEVEN, r, Y, M, C0, x0, init, True, dtype=dtype, kernel=1, want_grad=True, dynamics=_capi.DYN_COS,
                      ll_student=ll_student)
    assert one[4]["kernel"] == "direct"
    got = res["grad"][0].sum(axis=0)
    assert relerr(got, one[3]["grad"]) < (1e-11 if tag == "f64" else tol)
    ref = _grad_reference(_rounded(Y, tag), M, _rounded(C0, tag), x0, init, ll_student, D_UNEVEN)
    assert relerr(got, ref) < tol
    _close(res)


@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_loglik_sharded(r, tag, ll_student):
    dtype, tol = _dtype(tag)
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=2700 + r)
    init = impute_init(r)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, loglik=True, ll_student=ll_student)
    _check_ranks(res, dead, C0, tag)
    _compare(_whole(res), _oracle(Y, M, C0, x0, init, po.OracleConfig(robust=True), tag), tol)
    nll, lp = _loglik_reference(_rounded(Y, tag), M, _rounded(C0, tag), x0, init, True, ll_student)
    sc = res["scal"][0]
    assert sc.shape == (T, 10)
    assert relerr(sc[:, 8], nll) < tol and relerr(sc[:, 9], lp) < tol
    _close(res)


@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_linear_grad_sharded(r, tag, ll_student):
    """PSMF_GRAD_LINEAR: G_A and G_c of each one-step launch, summed by the caller, against the restatement on the
    oracle's trajectory (masked form: n = n_obs, q and C'Me over the observed rows)."""
    from rpsmf_b200 import _capi
    dtype, tol = _dtype(tag)
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=2800 + r)
    init = impute_init(r)
    A, c = _dynamics(r, seed=r)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, A=A, c=c, want_grad=True, dynamics=_capi.DYN_LINEAR,
                       grad_linear=True, ll_student=ll_student)
    _check_ranks(res, dead, C0, tag)
    cfg = po.OracleConfig(robust=True, dynamics=po.DYN_LINEAR, lin_A=A, lin_c=c)
    _compare(_whole(res), _oracle(Y, M, C0, x0, init, cfg, tag), tol)
    g = res["grad"][0].sum(axis=0)
    rGA, rGc = _linear_grad_reference(_rounded(Y, tag), M, _rounded(C0, tag), x0, init, A, c, True, ll_student)
    assert relerr(g[: r * r].reshape(r, r), rGA) < tol and relerr(g[r * r:], rGc) < tol
    _close(res)


def _tanh_dynamics(r):
    A = 0.9 * np.eye(r) + 0.1 * np.random.RandomState(r).randn(r, r) / np.sqrt(r)

    def f(x):
        xbar = np.tanh(A @ x)
        return xbar, (1.0 - xbar ** 2)[:, None] * A
    return f


def _external_one_engine(d, r, Y, M, C0, x0, init, f, dtype, exchange="nvlink", split=False, want_grad=True):
    """One engine over the whole series under external dynamics, one step per launch (run, or run_split with the identity
    all-reduce): X (T, r), Yrec (T, d), the per-step gradient d ell / d f, the state."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    eng = FilterEngine(d, r, dtype=dtype, robust=True, kernel=1, dynamics=_capi.DYN_EXTERNAL, exchange=exchange)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd = _padded(Y[None], dtype, eng.device)[0][0]
    Md = torch.as_tensor(M).to(eng.device)
    X, Yrec, G = np.zeros((T, r)), np.zeros((T, d)), np.zeros((T, r))
    x = x0.copy()
    for t in range(T):
        xbar, F = f(x)
        kw = dict(k0=1 + t, want_X=True, want_Yrec=True, want_grad=want_grad, xbar=xbar, F=F)
        out = eng.run_split(Yd[t:t + 1], Md[t:t + 1], allreduce=lambda buf: None, **kw) if split else eng.run(Yd[t:t + 1], Md[t:t + 1], **kw)
        assert eng.status() == -1
        X[t] = out["X"].cpu().numpy().reshape(r)
        Yrec[t] = out["Yrec"].double().cpu().numpy().reshape(d)
        if want_grad:
            G[t] = out["grad"].cpu().numpy().reshape(r)
        x = X[t]
    st = {k: (v.double().cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()}
    assert eng.launch_info()["kernel"] == "direct"
    eng.close()
    return X, Yrec, G, st


@pytest.mark.parametrize("r,tag", FLAG_RT, ids=FLAG_IDS)
def test_external_dynamics_sharded(r, tag):
    """PSMF_DYN_EXTERNAL (x_bar = tanh(A x), F its Jacobian, from the host every step): X, Yrec, the per-step gradient
    d ell / d f and C within 1e-12 of one engine on the whole series with the in-kernel exchange, one step per launch
    (fp32 storage: within the fp32 tolerance -- a last-bit difference of a reduction rounds a stored float differently)."""
    from rpsmf_b200 import _capi
    dtype, tol = _dtype(tag)
    lim = 1e-12 if tag == "f64" else tol
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=2900 + r)
    init = impute_init(r)
    f = _tanh_dynamics(r)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, want_grad=True, dynamics=_capi.DYN_EXTERNAL, xbar_fn=f)
    _check_ranks(res, dead, C0, tag)
    X, Yrec, scal, st, _ = _whole(res)
    oX, oYrec, oG, ost = _external_one_engine(D_UNEVEN, r, Y, M, C0, x0, init, f, dtype)
    assert relerr(X, oX) < lim and relerr(Yrec, oYrec) < lim and relerr(res["grad"][0], oG) < lim
    for k in ("C", "P", "V", "Q", "rho", "lam"):
        assert relerr(st[k], ost[k]) < lim, k
    _close(res)


# ---- 4. split == fused at world size 1 ------------------------------------------------------------------------------------
@pytest.mark.parametrize("ctas", [1, 3, 20])
@pytest.mark.parametrize("r", RANKS, ids=lambda r: "r%d" % r)
def test_split_equals_fused_world_one(r, ctas):
    """The external engine with the identity all-reduce, one step per launch pair, against the fused direct-load kernel
    over the same 12 steps in one launch: X, Yrec, the scalar record, C and the state are equal in value.  The fused pass
    applies the previous step's rank-1 update to a row as fma(e, g, c) before it takes that row's statistics; the split
    path applies the same fma at the end of phase 2 and reads the stored row in the next phase 1, which in fp64 is the
    same number.  (In fp32 it is not: the fused pass works on the updated row before it is rounded to float; the fp32
    sharded cells above hold the oracle tolerance.)"""
    d = 1000
    Y, M, C0, x0, dead = _problem("uneven1000", r, seed=3000 + r)
    init = impute_init(r)
    res = _sharded_run([(0, d)], r, Y, M, C0, x0, init, ctas=(ctas,))
    _check_ranks(res, dead, C0)
    assert res["info"][0]["ctas"] == ctas
    one = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=1, ctas=ctas)
    assert one[4]["kernel"] == "direct" and one[4]["ctas"] == ctas
    X, Yrec, scal, st, _ = _whole(res)
    assert np.array_equal(X, one[0])
    assert np.array_equal(Yrec, one[1])
    assert np.array_equal(scal, one[2])
    for k in ("C",) + REPLICATED:
        assert np.array_equal(st[k], one[3][k]), k
    _close(res)


# ---- 5. regressions of run_split and psmf_create ----------------------------------------------------------------------------
def test_run_split_writes_yrec():
    """run_split passes Yrec_out / want_Yrec to the pass (phase 1), which is the launch that writes the reconstruction:
    both give the fused kernel's Yrec, and the padding around a strided Yrec_out stays NaN."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    d, r = 1000, 9
    Y, M, C0, x0, _ = _problem("uneven1000", r, seed=3100)
    init = impute_init(r)
    one = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=1, ctas=3)
    for mode in ("out", "want"):
        eng = FilterEngine(d, r, robust=True, kernel=1, ctas=3, exchange="external")
        eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        Yd, Md = torch.as_tensor(Y).cuda(eng.device), torch.as_tensor(M).cuda(eng.device)
        Yrec, rec_buf = _padded(np.zeros((1, T, d)), torch.float64, eng.device, pad=5, fill=float("nan"))
        got = np.zeros((T, d))
        for t in range(T):
            if mode == "out":
                out = eng.run_split(Yd[t:t + 1], Md[t:t + 1], 1 + t, lambda buf: None, Yrec_out=Yrec[0, t:t + 1])
            else:
                out = eng.run_split(Yd[t:t + 1], Md[t:t + 1], 1 + t, lambda buf: None, want_Yrec=True)
            got[t] = out["Yrec"].cpu().numpy().reshape(d)
        assert eng.status() == -1
        eng.close()
        assert np.array_equal(got, one[1]), mode
        if mode == "out":
            assert np.array_equal(Yrec[0].cpu().numpy(), one[1])
            keep = torch.ones_like(rec_buf, dtype=torch.bool)
            keep.as_strided(Yrec.shape, Yrec.stride()).fill_(False)
            assert bool(rec_buf[keep].isnan().all())


def test_run_split_external_dynamics():
    """run_split on an engine with external dynamics hands x_bar and F to both launches: X, Yrec, the per-step
    gradient and the state equal those of run() with the in-kernel exchange, one step per launch."""
    torch = _torch()
    d, r = 1000, 9
    Y, M, C0, x0, _ = _problem("uneven1000", r, seed=3200)
    init = impute_init(r)
    f = _tanh_dynamics(r)
    a = _external_one_engine(d, r, Y, M, C0, x0, init, f, torch.float64)
    b = _external_one_engine(d, r, Y, M, C0, x0, init, f, torch.float64, exchange="external", split=True)
    for i in range(3):
        assert np.array_equal(a[i], b[i]), i
    for k in ("C",) + REPLICATED[:-1]:
        assert np.array_equal(a[3][k], b[3][k]), k


def test_rho_vector_with_external_exchange_refused_at_create():
    """A non-uniform diagonal R has a longer statistics vector than the caller-driven exchange carries; the pair is
    refused when the engine is created (nothing is launched)."""
    from rpsmf_b200 import FilterEngine, _capi
    for r in (1, 12, 16):
        for loglik in (False, True):
            with pytest.raises(_capi.PsmfError, match="PSMF_RHO_VECTOR"):
                FilterEngine(1000, r, rho_vector=True, exchange="external", loglik=loglik)


# ---- 6. the first-bad-step report on every rank -------------------------------------------------------------------------------
def test_status_reports_the_bad_step_on_every_rank():
    """An inf in rank 1's rows at step 5 (a data value): every rank reports no bad step after steps 0..4, and after step 5
    every rank reports 0, the bad step of its last one-step run -- the statistics are summed, so the replicated update of
    every rank sees it, not only the rank that holds the row."""
    r = 9
    Y, M, C0, x0, _ = _problem("uneven1000", r, seed=3300)
    Y[5, 7] = np.inf
    M[5, 7] = 1
    init = impute_init(r)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, steps=6)
    assert (res["status"][:5] == -1).all(), res["status"]
    assert (res["status"][5] == 0).all(), res["status"]
    _close(res)


# ---- 7. forecast and evaluation tools on shards ------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", [1, 9, 16], ids=lambda r: "r%d" % r)
def test_tools_on_shards(r, tag):
    """After a sharded run under cos dynamics, the forecast and the evaluation of each rank against one engine that holds
    the same state for the whole series (the concatenated C, the replicated x and theta).  predict: Xpred bit-identical on
    all ranks and equal to the one engine's, Ypred concatenated over the shards equal to the one engine's to 1e-12 (fp32
    output: within one ulp).  eval_full per shard: the sums over the ranks match the one-engine sum to 1e-12 and the
    counts exactly."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    dtype, _ = _dtype(tag)
    d = D_UNEVEN
    Y, M, C0, x0, _ = _problem("uneven1000", r, seed=3400 + r)
    init = impute_init(r)
    theta = _theta(r)
    res = _sharded_run(UNEVEN, r, Y, M, C0, x0, init, dtype=dtype, theta=theta, dynamics=_capi.DYN_COS)
    _check_ranks(res)
    st = _whole(res)[3]
    one = FilterEngine(d, r, dtype=dtype, robust=True, kernel=1, dynamics=_capi.DYN_COS)
    one.set_state(C_=st["C"], x=st["x"], theta=st["theta"])
    n_pred = 7
    Xp1, Yp1 = one.predict(n_pred, T + 1)
    Xp1, Yp1 = Xp1.cpu().numpy(), Yp1.double().cpu().numpy()
    Xps, Yps = [], []
    for eng in res["engines"]:
        Xp, Yp = eng.predict(n_pred, T + 1)
        Xps.append(Xp.cpu().numpy())
        Yps.append(Yp.double().cpu().numpy())
    for Xp in Xps:
        assert np.array_equal(Xp, Xp1)
    Ys = np.concatenate(Yps, axis=1)
    if tag == "f64":
        assert relerr(Ys, Yp1) < 1e-12
    else:
        assert np.all(np.abs(Ys - Yp1) <= np.spacing(np.abs(Yp1).astype(np.float32)).astype(np.float64))
    rng = np.random.RandomState(r)
    Yorig = Y + rng.randn(T, d)
    E = ((rng.rand(T, d) < 0.15) & (M == 0)).astype(np.uint8)
    E[:, 0] = 1                                                          # the 1-row shard takes part
    Xs = torch.as_tensor(res["X"][0]).to(one.device)
    tot = np.zeros(2)
    for (b, e), eng in zip(UNEVEN, res["engines"]):
        Yo = _padded(np.ascontiguousarray(Yorig[None, :, b:e]), dtype, eng.device)[0][0]
        Ed = torch.as_tensor(np.ascontiguousarray(E[:, b:e])).to(eng.device)
        tot += eng.eval_full(Xs, Yo, Ed).cpu().numpy().reshape(2)
    Yo1 = _padded(Yorig[None], dtype, one.device)[0][0]
    ref = one.eval_full(Xs, Yo1, torch.as_tensor(E).to(one.device)).cpu().numpy().reshape(2)
    assert tot[1] == ref[1] == E.sum()
    assert abs(tot[0] - ref[0]) <= 1e-12 * ref[0]
    one.close()
    _close(res)


# ---- 8. the emulation against the NVLink mailboxes ---------------------------------------------------------------------------
def test_emulation_matches_the_in_kernel_exchange():
    """Two ranks on one GPU exchange through each other's mailboxes (CUDA IPC); rank 0 then runs the two-engine external
    emulation of this file in its own process: X, the scalar record, the state and each shard's C are equal in value."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "tests", "multi_gpu_external_check.py"), "--same-device"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, PSMF_SPIN_TIMEOUT_MS="60000"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" OK") == 4 and "FAIL" not in r.stdout, r.stdout[-3000:]
