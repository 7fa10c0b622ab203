# -*- coding: utf-8 -*-
"""Gradient of the summed incremental log-likelihood with respect to A and c under linear dynamics x_bar = A x + c
(PSMF_GRAD_LINEAR), on every filter kernel.

The kernels accumulate G_A = sum_k gf_k x_{k-1}' and G_c = sum_k gf_k, gf_k = d ell_k / d x_bar_k with N, eta and V held
fixed (the convention of the cos gradient).  Each case forces its kernel and checks from launch_info() that the variant it
meant to test ran.  Without a mask the sums are compared with a float64 restatement built on the oracle's trajectory; with
a mask every kernel must agree to 1e-11 and match the same restatement over the observed rows (n = n_obs, q and C'Me over
them), which pins the masked form against nothing but itself, as for the cos gradient."""

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _padded, _torch
from test_gpu_kernel_matrix import KNAME, KERNEL_KW, FLAG_D, SPLIT_RANKS, TOL32, _check_variant, _stream_d

pytestmark = pytest.mark.gpu

T = 12
CHUNKS = [0, 5, 12]                # two launches: the gradient of each launch is summed over that launch only
RANKS = [1, 5, 8, 9, 16]
VARIANTS = {
    # name: (kernel, d, S, engine keywords); d is a function of (r, esize) for the streaming TMA variant
    "direct": (1, 4001, None, {}),
    "tma_resident": (2, 1600, None, dict(ctas=2)),
    "tma_stream": (2, _stream_d, None, dict(ctas=1)),
    "batch8": (3, 1100, 3, {}),
    "batch4": (3, 203, 3, {}),
}
MODELS = {"psmf_gauss": (False, False), "psmf_student": (False, True), "rpsmf_gauss": (True, False), "rpsmf_student": (True, True)}


def _dynamics(r, seed, with_c=True):
    """A stable, non-symmetric A and an offset c."""
    rng = np.random.RandomState(seed)
    A = 0.9 * np.eye(r) + 0.1 * rng.randn(r, r) / np.sqrt(r)
    return A, (0.1 * rng.randn(r) if with_c else None)


def _linear_grad_reference(Y, M, C0, x0, init, A, c, robust, ll_student, simplified=False):
    """(G_A, G_c) from the oracle's trajectory: step k uses the C, V, lambda and x_{k-1} entering it and its own eta."""
    d = C0.shape[0]
    cfg = po.OracleConfig(robust=robust, simplified=simplified, c_update_transpose=True, dynamics=po.DYN_LINEAR, lin_A=A, lin_c=c)
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"], init["lam"])
    r = x0.shape[0]
    GA, Gc = np.zeros((r, r)), np.zeros(r)
    for t in range(Y.shape[0]):
        m = np.ones(d) if M is None else M[t].astype(float)
        new, out = po.step(st, cfg, Y[t], m, k=1 + t)
        f = out["xbar"]
        e = m * (Y[t] - st.C @ f)
        gf = po.dll_df(ll_student, f, st.V, st.C.T @ e, float(e @ e), out["eta"], st.lam, float(m.sum()))
        GA += np.outer(gf, st.x)
        Gc += gf
        st = new
    return GA, Gc


def _run(d, r, Y, M, C0, x0, init, A, c, robust=True, S=None, chunks=CHUNKS, dtype=None, **kw):
    """Filter Y (T, d) or (S, T, d) in the launches given by `chunks`; returns (G_A, G_c) summed over the launches (with
    the series axis when S is given), X and launch_info."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    dtype = dtype or torch.float64
    eng = FilterEngine(d, r, dtype=dtype, robust=robust, n_series=S or 1, dynamics=_capi.DYN_LINEAR, grad_linear=True,
                       c_update_transpose=True, **kw)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    eng.set_linear_dynamics(A, c)
    one = S is None
    Yd = _padded(Y[None] if one else Y, dtype, eng.device)[0]
    Md = None if M is None else _padded(M[None] if one else M, torch.uint8, eng.device)[0]
    GA, Gc, Xs = 0.0, 0.0, []
    for a, b in zip(chunks[:-1], chunks[1:]):
        out = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, want_grad=True)
        assert eng.status() == -1
        GA = GA + out["grad_A"].cpu().numpy()
        Gc = Gc + out["grad_c"].cpu().numpy()
        Xs.append(out["X"].reshape(S or 1, b - a, r).cpu().numpy())
    info = eng.launch_info()
    eng.close()
    X = np.concatenate(Xs, axis=1)
    return GA, Gc, (X[0] if one else X), info


def _rounded(a, f32):
    return a.astype(np.float32).astype(np.float64) if f32 else a


ORACLE_PARAMS = [(v, r, "f64", m) for v in VARIANTS for r in RANKS for m in MODELS] + \
                [(v, r, "f32", "rpsmf_gauss") for v in VARIANTS for r in RANKS]


@pytest.mark.parametrize("name,r,tag,model", ORACLE_PARAMS, ids=["%s-r%d-%s-%s" % p for p in ORACLE_PARAMS])
def test_linear_grad_against_oracle(name, r, tag, model):
    torch = _torch()
    kernel, d, S, kw = VARIANTS[name]
    f32 = tag == "f32"
    esize = 4 if f32 else 8
    if callable(d):
        d = d(r, esize)
    robust, ll_student = MODELS[model]
    Y, _, C0, x0 = make_problem(d, r, T, seed=300 + 7 * r + d % 89, missing=0.0, S=S)
    init = impute_init(r)
    A, c = _dynamics(r, seed=r)
    GA, Gc, _, info = _run(d, r, Y, None, C0, x0, init, A, c, robust=robust, S=S, ll_student=ll_student, kernel=kernel,
                           dtype=torch.float32 if f32 else torch.float64, **kw)
    _check_variant(name, info, r, esize, d)
    tol = TOL32 if f32 else TOL
    for s in range(S or 1):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        rGA, rGc = _linear_grad_reference(_rounded(one(Y), f32), None, _rounded(one(C0), f32), one(x0), init, A, c, robust, ll_student)
        assert relerr(one(GA), rGA) < tol
        assert relerr(one(Gc), rGc) < tol


MASK_CASES = ["byte", "nan", "simplified", "no_c"]


@pytest.mark.parametrize("case", MASK_CASES)
@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("r", SPLIT_RANKS, ids=lambda r: "r%d" % r)
def test_linear_grad_masked_kernels_agree(r, ll_student, case):
    d = FLAG_D
    Y, M, C0, x0 = make_problem(d, r, T, seed=500 + r)
    M[:, [1, d // 2]] = 0
    Y = Y * M
    init = impute_init(r)
    A, c = _dynamics(r, seed=r, with_c=case != "no_c")
    simplified = case == "simplified"
    Yk, Mk, kw = Y, M, dict(ll_student=ll_student, simplified=simplified)
    if case == "nan":
        Yk = Y.copy()
        Yk[M == 0] = np.nan
        Mk, kw["nan_mask"] = None, True
    got = []
    for kernel in (1, 2, 3):
        GA, Gc, _, info = _run(d, r, Yk, Mk, C0, x0, init, A, c, **kw, **KERNEL_KW[kernel])
        assert info["kernel"] == KNAME[kernel]
        got.append((GA, Gc))
    for GA, Gc in got[1:]:
        assert relerr(GA, got[0][0]) < 1e-11 and relerr(Gc, got[0][1]) < 1e-11
    rGA, rGc = _linear_grad_reference(Y, M, C0, x0, init, A, c, True, ll_student, simplified)
    assert relerr(got[0][0], rGA) < TOL and relerr(got[0][1], rGc) < TOL


@pytest.mark.parametrize("r", [1, 5, 9, 16], ids=lambda r: "r%d" % r)
@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
def test_linear_grad_matches_external_path(r, ll_student):
    """The same problem through the external-dynamics path, one step per launch with x_bar = A x + c and F = A: the sum of
    the per-step d ell / d f times x_{k-1}' is the in-kernel G_A."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d = FLAG_D
    Y, M, C0, x0 = make_problem(d, r, T, seed=700 + r)
    Y = Y * M
    init = impute_init(r)
    A, c = _dynamics(r, seed=r)
    GA, Gc, X, info = _run(d, r, Y, M, C0, x0, init, A, c, ll_student=ll_student, kernel=1, ctas=3, chunks=[0, T])
    assert info["kernel"] == "direct"
    eng = FilterEngine(d, r, robust=True, dynamics=_capi.DYN_EXTERNAL, ll_student=ll_student, c_update_transpose=True,
                       kernel=1, ctas=3)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd = torch.as_tensor(Y).cuda(eng.device)
    Md = torch.as_tensor(M).cuda(eng.device)
    eGA, eGc, x = np.zeros((r, r)), np.zeros(r), x0.copy()
    for t in range(T):
        out = eng.run(Yd[t:t + 1], Md[t:t + 1], k0=1 + t, want_X=True, want_grad=True, xbar=A @ x + c, F=A)
        g = out["grad"].cpu().numpy()
        eGA += np.outer(g, x)
        eGc += g
        x = out["X"].cpu().numpy().reshape(r)
    assert eng.status() == -1
    eng.close()
    assert relerr(GA, eGA) < 1e-12 and relerr(Gc, eGc) < 1e-12


def test_linear_grad_batch_of_series():
    """Six series in one batch launch: every series' gradient against its own restatement."""
    d, r, S = 512, 8, 6
    Y, M, C0, x0 = make_problem(d, r, T, seed=11, S=S)
    Y = Y * M
    init = impute_init(r)
    A, c = _dynamics(r, seed=3)
    GA, Gc, _, info = _run(d, r, Y, M, C0, x0, init, A, c, S=S)
    assert info["kernel"] == "batch" and GA.shape == (S, r, r) and Gc.shape == (S, r)
    for s in range(S):
        rGA, rGc = _linear_grad_reference(Y[s], M[s], C0[s], x0[s], init, A, c, True, False)
        assert relerr(GA[s], rGA) < TOL and relerr(Gc[s], rGc) < TOL


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
def test_linear_grad_bit_identical_runs(kernel):
    d, r = FLAG_D, 9
    Y, M, C0, x0 = make_problem(d, r, T, seed=13)
    Y = Y * M
    init = impute_init(r)
    A, c = _dynamics(r, seed=5)
    a = _run(d, r, Y, M, C0, x0, init, A, c, **KERNEL_KW[kernel])
    b = _run(d, r, Y, M, C0, x0, init, A, c, **KERNEL_KW[kernel])
    assert a[3]["kernel"] == KNAME[kernel]
    for i in range(3):
        assert np.array_equal(a[i], b[i])


def test_linear_grad_does_not_change_the_filter():
    """The flag adds the gradient and nothing else: X is bit for bit that of the engine without it."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r = FLAG_D, 8
    Y, M, C0, x0 = make_problem(d, r, T, seed=17)
    Y = Y * M
    init = impute_init(r)
    A, c = _dynamics(r, seed=7)
    for kernel in (1, 2, 3):
        _, _, X, info = _run(d, r, Y, M, C0, x0, init, A, c, chunks=[0, T], **KERNEL_KW[kernel])
        eng = FilterEngine(d, r, robust=True, dynamics=_capi.DYN_LINEAR, c_update_transpose=True, **KERNEL_KW[kernel])
        eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        eng.set_linear_dynamics(A, c)
        out = eng.run(torch.as_tensor(Y).cuda(eng.device), torch.as_tensor(M).cuda(eng.device), want_X=True)
        assert eng.launch_info()["kernel"] == info["kernel"] == KNAME[kernel]
        assert np.array_equal(out["X"].cpu().numpy(), X)
        eng.close()


def test_grad_linear_needs_linear_dynamics():
    from rpsmf_b200 import FilterEngine, _capi
    for dyn in (_capi.DYN_IDENTITY, _capi.DYN_COS, _capi.DYN_EXTERNAL):
        with pytest.raises(_capi.PsmfError, match="PSMF_DYN_LINEAR"):
            FilterEngine(64, 4, dynamics=dyn, grad_linear=True)


# ---- class surface: a marked affine callable runs as device linear dynamics -------------------------------------------
def _affine_fn(r):
    B = 0.05 * np.random.RandomState(r).randn(r, r)

    def f(theta, x, t):
        th = theta.reshape(-1)
        A = 0.85 * np.eye(r) + 0.1 * np.diag(np.sin(th)) + B
        return A @ x + (0.2 * th * th).reshape(r, 1)
    return f


def _ydict(Y):
    return {k + 1: Y[k].reshape(-1, 1) for k in range(Y.shape[0])}


def _make_class(kind, fn, theta0, C0, x0, T):
    from rpsmf_b200 import PSMFIter, PSMFRecursive, rPSMFIter
    d, r = C0.shape
    Q, R = 0.05 * np.eye(r), 2.0 * np.eye(d)
    if kind == "rpsmf":
        return rPSMFIter(theta0.copy(), C0, 0.5 * np.eye(r), x0.reshape(r, 1), np.eye(r), Q, R, 1.8, fn)
    cls = PSMFRecursive if kind == "recursive" else PSMFIter
    return cls(theta0.copy(), C0, 0.5 * np.eye(r), x0.reshape(r, 1), np.eye(r), {k: Q for k in range(T + 1)},
               {k: R for k in range(T + 1)}, fn)


def _count_runs(o):
    eng = o._get_engine()
    calls = []
    run = eng.run

    def counted(*a, **k):
        calls.append(1)
        return run(*a, **k)
    eng.run = counted
    return calls


@pytest.mark.parametrize("kind", ["psmf", "rpsmf"])
def test_classes_marked_affine_matches_external_path(kind):
    from rpsmf_b200 import _capi
    from rpsmf_b200.nonlinearities import affine
    d, r, T, n_iter = 40, 4, 30, 4
    Y, _, C0, x0 = make_problem(d, r, T, seed=23, missing=0.0)
    theta0 = 0.3 + 0.1 * np.arange(r).reshape(r, 1)
    fn = _affine_fn(r)
    a, b = _make_class(kind, affine(fn), theta0, C0, x0, T), _make_class(kind, fn, theta0, C0, x0, T)
    assert a._dyn == _capi.DYN_LINEAR and b._dyn == _capi.DYN_EXTERNAL
    calls = _count_runs(a)
    y = _ydict(Y)
    a.optim_init(gam=1e-2)
    b.optim_init(gam=1e-2)
    for i in range(1, n_iter + 1):
        a.step(y, i, T)
        b.step(y, i, T)
        assert len(calls) == i                                   # one filter launch per sweep
        assert np.max(np.abs(a._gradsum)) > 0 and relerr(a._gradsum, b._gradsum) < 1e-9
        a.predict(i, T, 5)
        b.predict(i, T, 5)
        a.optim_update(i)
        b.optim_update(i)
        assert relerr(a._theta[i], b._theta[i]) < 1e-9
    assert relerr(a._mu[T], b._mu[T]) < 1e-9 and relerr(a._C[T], b._C[T]) < 1e-9
    for k in list(range(1, T + 6)):
        assert relerr(a._y_pred[k], b._y_pred[k]) < 1e-9, k
    a.close(); b.close()


@pytest.mark.parametrize("ue", [1, 7])
def test_recursive_marked_affine_matches_external_path(ue):
    from rpsmf_b200.nonlinearities import affine
    d, r, T = 40, 4, 30
    Y, _, C0, x0 = make_problem(d, r, T, seed=29, missing=0.0)
    theta0 = 0.3 + 0.1 * np.arange(r).reshape(r, 1)
    fn = _affine_fn(r)
    a, b = _make_class("recursive", affine(fn), theta0, C0, x0, T), _make_class("recursive", fn, theta0, C0, x0, T)
    calls = _count_runs(a)
    y = _ydict(Y)
    a.run(y, T, 5, update_every=ue)
    b.run(y, T, 5, update_every=ue)
    assert len(calls) == -(-T // ue)                             # one launch per update_every block
    for k in range(1, T + 1):
        assert relerr(a._theta[k], b._theta[k]) < 1e-9, k
    assert relerr(a._mu[T], b._mu[T]) < 1e-9 and relerr(a._C[T], b._C[T]) < 1e-9
    for k in range(1, T + 6):
        assert relerr(a._y_pred[k], b._y_pred[k]) < 1e-9, k
    a.close(); b.close()


def test_marked_callable_that_is_not_affine_raises():
    from rpsmf_b200.nonlinearities import affine
    d, r, T = 40, 3, 5
    Y, _, C0, x0 = make_problem(d, r, T, seed=31, missing=0.0)
    for fn in (lambda th, x, t: np.tanh(x), lambda th, x, t: 0.9 * x + 0.01 * t):
        o = _make_class("psmf", affine(fn), np.ones((r, 1)), C0, x0, T)
        with pytest.raises(ValueError, match="affine"):
            o.step(_ydict(Y), 1, T)
        o.close()


def test_row_sharded_ranks_share_one_gpu():
    """Two row-sharded ranks on cuda:0 (the same-device mechanism of tests/multi_gpu_check.py): G_A and G_c bit-identical
    on both ranks and within 1e-9 of the one-GPU engine, on the direct-load and the TMA-staged kernel."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29521", os.path.join(root, "tests", "multi_gpu_linear_grad_check.py"), "--same-device"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, PSMF_SPIN_TIMEOUT_MS="60000"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" OK") == 4 and "FAIL" not in r.stdout
