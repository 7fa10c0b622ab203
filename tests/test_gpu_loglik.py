# -*- coding: utf-8 -*-
"""Per-step learning objective and one-step predictive log-density (PSMF_LOGLIK) on every filter kernel.

Each case forces its kernel and checks from launch_info() that the variant it meant to test ran.  The kernels' nll_k and
log p_k are compared per step with the float64 restatement of tests/loglik_oracle.py on the oracle's trajectory (fp64 1e-9,
fp32 storage 1e-4 on fp32-rounded Y and C0); that restatement is itself checked against dense densities and against the
gradient in tests/test_loglik_cpu.py."""

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from loglik_oracle import run_loglik, step_loglik
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _padded, _torch
from test_gpu_kernel_matrix import FLAG_D, KERNEL_KW, KNAME, SPLIT_RANKS, TOL32, VARIANTS as KM_VARIANTS, _check_variant

pytestmark = pytest.mark.gpu

T = 12
CHUNKS = [0, 5, 12]                # two launches: the record of each launch covers its own steps
RANKS = [1, 5, 8, 9, 16]
VARIANTS = {k: KM_VARIANTS[k] for k in ("direct", "direct_S3", "rhovec", "tma_resident", "tma_stream", "batch8", "batch4")}
MODELS = {"psmf_gauss": (False, False), "psmf_student": (False, True), "rpsmf_gauss": (True, False), "rpsmf_student": (True, True)}


def _init(r, d, rho_vector, seed=0):
    init = impute_init(r)
    if rho_vector:
        init["rho"] = 10.0 * (0.5 + np.random.RandomState(seed).rand(d))
    return init


def _engine(d, r, init, C0, x0, S=None, loglik=True, A=None, c=None, theta=None, **kw):
    from rpsmf_b200 import FilterEngine
    eng = FilterEngine(d, r, n_series=S or 1, c_update_transpose=True, loglik=loglik, **kw)
    rho = init["rho"]
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=rho if np.ndim(rho) else [rho], lam=[init["lam"]],
                  theta=theta)
    if A is not None:
        eng.set_linear_dynamics(A, c)
    return eng


def _run(d, r, Y, M, C0, x0, init, S=None, chunks=CHUNKS, dtype=None, loglik=True, want_grad=False, A=None, c=None, theta=None,
         nan=False, **kw):
    """Filter Y (T, d) or (S, T, d) in the launches given by `chunks`.  Returns dict(scal (S?, T, 8 or 10), X, grad (summed
    over the launches), state, info)."""
    torch = _torch()
    dtype = dtype or torch.float64
    eng = _engine(d, r, init, C0, x0, S=S, loglik=loglik, A=A, c=c, theta=theta, dtype=dtype, nan_mask=nan, **kw)
    one = S is None
    Yh = Y[None] if one else Y
    if nan:
        Yh = np.where((M[None] if one else M) == 0, np.nan, Yh)
    Yd = _padded(Yh, dtype, eng.device)[0]
    Md = None if (M is None or nan) else _padded(M[None] if one else M, torch.uint8, eng.device)[0]
    scal, X, grad = [], [], 0.0
    for a, b in zip(chunks[:-1], chunks[1:]):
        out = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, want_scal=True, want_grad=want_grad)
        assert eng.status() == -1
        scal.append(out["scal"].reshape(S or 1, b - a, -1).cpu().numpy())
        X.append(out["X"].reshape(S or 1, b - a, r).cpu().numpy())
        if want_grad:
            g = out["grad_A"] if "grad_A" in out else out["grad"]
            grad = grad + np.concatenate([g.reshape(S or 1, -1).cpu().numpy()] +
                                         ([out["grad_c"].reshape(S or 1, -1).cpu().numpy()] if "grad_c" in out else []), axis=1)
    st = {k: (v.cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()}
    info = eng.launch_info()
    eng.close()
    res = dict(scal=np.concatenate(scal, axis=1), X=np.concatenate(X, axis=1), grad=grad, state=st, info=info)
    if one:
        res["scal"], res["X"] = res["scal"][0], res["X"][0]
    return res


def _reference(Y, M, C0, x0, init, robust, ll_student, simplified=False, dynamics=po.DYN_IDENTITY, A=None, c=None, theta=None):
    cfg = po.OracleConfig(robust=robust, simplified=simplified, c_update_transpose=True, dynamics=dynamics, lin_A=A, lin_c=c)
    rho = init["rho"]
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(),
                        rho if np.ndim(rho) == 0 else np.array(rho), init["lam"], None if theta is None else np.asarray(theta, float))
    return run_loglik(st, cfg, Y, M, ll_student)[1:]


def _rounded(a, f32):
    return a.astype(np.float32).astype(np.float64) if f32 else a


def _masked(d, r, S, seed):
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, S=S)
    M[..., [1, d // 2]] = 0
    M[..., T - 1, :] = 0       # a step with every row missing, the last: the oracle's robust phi is NaN after it (0 * inf)
    return Y * M, M, C0, x0


def _check(scal, Y, M, C0, x0, init, robust, ll_student, tol, S=None, f32=False, **kw):
    for s in range(S or 1):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        nll, lp = _reference(_rounded(one(Y), f32), one(M), _rounded(one(C0), f32), one(x0), init, robust, ll_student, **kw)
        sc = one(scal)
        assert sc.shape[-1] == 10
        assert relerr(sc[:, 8], nll) < tol, (sc[:, 8], nll)
        assert relerr(sc[:, 9], lp) < tol, (sc[:, 9], lp)
        assert sc[T - 1, 8] == 0.0 and sc[T - 1, 9] == 0.0         # every row missing: no term


ORACLE_PARAMS = [(v, r, "f64", m) for v in VARIANTS for r in RANKS for m in MODELS] + \
                [(v, r, "f32", "rpsmf_student") for v in VARIANTS for r in RANKS]


@pytest.mark.parametrize("name,r,tag,model", ORACLE_PARAMS, ids=["%s-r%d-%s-%s" % p for p in ORACLE_PARAMS])
def test_loglik_against_oracle(name, r, tag, model):
    torch = _torch()
    kernel, d, S, kw = VARIANTS[name]
    f32 = tag == "f32"
    esize = 4 if f32 else 8
    if callable(d):
        d = d(r, esize)
    robust, ll_student = MODELS[model]
    Y, M, C0, x0 = _masked(d, r, S, seed=900 + 7 * r + d % 89)
    init = _init(r, d, kw.get("rho_vector", False))
    res = _run(d, r, Y, M, C0, x0, init, S=S, robust=robust, ll_student=ll_student, kernel=kernel,
               dtype=torch.float32 if f32 else torch.float64, **kw)
    _check_variant(name, res["info"], r, esize, d)
    _check(res["scal"], Y, M, C0, x0, init, robust, ll_student, TOL32 if f32 else TOL, S=S, f32=f32)


def _dynamics(r, seed):
    rng = np.random.RandomState(seed)
    return 0.9 * np.eye(r) + 0.1 * rng.randn(r, r) / np.sqrt(r), 0.1 * rng.randn(r)


FLAG_CASES = ["nan", "simplified", "cos", "linear"]


@pytest.mark.parametrize("case", FLAG_CASES)
@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("r", SPLIT_RANKS, ids=lambda r: "r%d" % r)
def test_loglik_flags_on_each_kernel(r, kernel, ll_student, case):
    from rpsmf_b200 import _capi
    d = FLAG_D
    Y, M, C0, x0 = _masked(d, r, None, seed=1200 + r)
    init = impute_init(r)
    kw = dict(robust=True, ll_student=ll_student, **KERNEL_KW[kernel])
    ref_kw = {}
    if case == "nan":
        a = _run(d, r, Y, M, C0, x0, init, **kw)
        b = _run(d, r, Y, M, C0, x0, init, nan=True, **kw)
        assert a["info"]["kernel"] == b["info"]["kernel"] == KNAME[kernel]
        assert np.array_equal(a["scal"], b["scal"]) and np.array_equal(a["X"], b["X"])
        res = a
    else:
        if case == "simplified":
            kw["simplified"] = ref_kw["simplified"] = True
        elif case == "cos":
            kw["dynamics"] = ref_kw["dynamics"] = _capi.DYN_COS
            kw["theta"] = ref_kw["theta"] = 0.05 + 0.01 * np.arange(r)
        else:
            kw["dynamics"] = ref_kw["dynamics"] = _capi.DYN_LINEAR
            A, c = _dynamics(r, seed=r)
            kw["A"] = ref_kw["A"] = A
            kw["c"] = ref_kw["c"] = c
        res = _run(d, r, Y, M, C0, x0, init, **kw)
        assert res["info"]["kernel"] == KNAME[kernel]
    _check(res["scal"], Y, M, C0, x0, init, True, ll_student, TOL, **ref_kw)


@pytest.mark.parametrize("robust", [False, True], ids=["psmf", "rpsmf"])
@pytest.mark.parametrize("r", [1, 9])
def test_loglik_external_dynamics(r, robust):
    """One step per launch with x_bar and F from the host (the direct-load kernel): each step's record against the oracle."""
    torch = _torch()
    from rpsmf_b200 import _capi
    d = FLAG_D
    Y, M, C0, x0 = _masked(d, r, None, seed=1300 + r)
    init = impute_init(r)
    A, c = _dynamics(r, seed=r + 1)
    eng = _engine(d, r, init, C0, x0, robust=robust, ll_student=robust, dynamics=_capi.DYN_EXTERNAL, kernel=1, ctas=3)
    Yd, Md = torch.as_tensor(Y).cuda(eng.device), torch.as_tensor(M).cuda(eng.device)
    cfg = po.OracleConfig(robust=robust, c_update_transpose=True)
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"], init["lam"])
    x = x0.copy()
    for t in range(T):
        out = eng.run(Yd[t:t + 1], Md[t:t + 1], k0=1 + t, want_X=True, want_loglik=True, xbar=A @ x + c, F=A)
        st, _, nll, lp = step_loglik(st, cfg, Y[t], M[t], 1 + t, robust, xbar_F=(A @ st.x + c, A))
        got = (float(out["nll"][0]), float(out["logpred"][0]))
        if t == T - 1:
            assert got == (0.0, 0.0)
        else:
            assert abs(got[0] - nll) <= TOL * abs(nll) and abs(got[1] - lp) <= TOL * abs(lp), (t, got, nll, lp)
        x = out["X"].cpu().numpy().reshape(r)
    assert eng.launch_info()["kernel"] == "direct" and eng.status() == -1
    eng.close()


@pytest.mark.parametrize("robust", [False, True], ids=["psmf", "rpsmf"])
@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
def test_logdet_term_vanishes_without_pbar(kernel, robust):
    """P = Q = 0 makes Pbar = 0: I + Pbar G = I, every pivot is 1, and log p_k is the diagonal-S form computed here from the
    oracle's trajectory, to 1e-12."""
    from scipy.special import gammaln
    d, r = FLAG_D, 5
    Y, M, C0, x0 = _masked(d, r, None, seed=1400)
    init = dict(impute_init(r), P=np.zeros((r, r)), Q=np.zeros((r, r)))
    res = _run(d, r, Y, M, C0, x0, init, robust=robust, **KERNEL_KW[kernel])
    assert res["info"]["kernel"] == KNAME[kernel]
    cfg = po.OracleConfig(robust=robust, c_update_transpose=True)
    st = po.OracleState(C0.copy(), x0.copy(), init["P"], init["V"].copy(), init["Q"], init["rho"], init["lam"])
    for t in range(T):
        lam = st.lam
        st, out = po.step(st, cfg, Y[t], M[t].astype(float), k=1 + t)
        obs = M[t] > 0
        n = float(obs.sum())
        if n == 0:
            assert res["scal"][t, 9] == 0.0
            continue
        ra = out["rho"] + out["a"]                                       # rho entering the step + a
        logdet = n * np.log(ra)
        d2 = float(np.sum(out["e"][obs] ** 2)) / ra
        if robust:
            ref = gammaln(0.5 * (lam + n)) - gammaln(0.5 * lam) - 0.5 * n * np.log(lam * np.pi) - 0.5 * logdet \
                - 0.5 * (lam + n) * np.log1p(d2 / lam)
        else:
            ref = -0.5 * (n * np.log(2.0 * np.pi) + logdet + d2)
        assert abs(res["scal"][t, 9] - ref) <= 1e-12 * abs(ref), (t, res["scal"][t, 9], ref)


@pytest.mark.parametrize("case", ["direct", "rhovec", "tma", "batch", "grad_cos", "grad_linear_direct", "grad_linear_tma",
                                  "grad_linear_batch"])
def test_loglik_does_not_perturb_the_filter(case):
    """X, entries 0..7 of the record, grad_out and the final state are bit for bit those of the engine without the flag;
    a repeat run with the flag gives the same bits."""
    from rpsmf_b200 import _capi
    d, r = FLAG_D, 9
    Y, M, C0, x0 = _masked(d, r, None, seed=1500)
    kernel = {"direct": 1, "rhovec": 1, "tma": 2, "batch": 3, "grad_cos": 1}.get(case, None)
    if kernel is None:
        kernel = {"direct": 1, "tma": 2, "batch": 3}[case.rsplit("_", 1)[1]]
    kw = dict(KERNEL_KW[kernel], robust=True, ll_student=True)
    init = _init(r, d, case == "rhovec")
    if case == "rhovec":
        kw["rho_vector"] = True
    if case == "grad_cos":
        kw.update(dynamics=_capi.DYN_COS, theta=0.05 + 0.01 * np.arange(r), want_grad=True)
    if case.startswith("grad_linear"):
        A, c = _dynamics(r, seed=2)
        kw.update(dynamics=_capi.DYN_LINEAR, A=A, c=c, grad_linear=True, want_grad=True)
    on = _run(d, r, Y, M, C0, x0, init, loglik=True, **kw)
    again = _run(d, r, Y, M, C0, x0, init, loglik=True, **kw)
    off = _run(d, r, Y, M, C0, x0, init, loglik=False, **kw)
    assert on["info"]["kernel"] == off["info"]["kernel"] == KNAME[kernel]
    assert on["scal"].shape[-1] == 10 and off["scal"].shape[-1] == 8
    assert np.array_equal(on["X"], off["X"]) and np.array_equal(on["scal"][..., :8], off["scal"])
    assert np.array_equal(np.asarray(on["grad"]), np.asarray(off["grad"]))
    if kw.get("want_grad"):
        assert np.max(np.abs(on["grad"])) > 0
    for k, v in off["state"].items():
        if v is not None:
            assert np.array_equal(on["state"][k], v), k
    assert np.array_equal(on["scal"], again["scal"]) and np.array_equal(on["X"], again["X"])
    assert np.all(np.isfinite(on["scal"][..., 8:]))


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
def test_loglik_without_scal_out(kernel):
    """The flag with no record requested: the run succeeds and filters exactly as without the flag."""
    torch = _torch()
    d, r = FLAG_D, 8
    Y, M, C0, x0 = _masked(d, r, None, seed=1600)
    init = impute_init(r)
    Xs = []
    for loglik in (True, False):
        eng = _engine(d, r, init, C0, x0, loglik=loglik, **KERNEL_KW[kernel])
        out = eng.run(torch.as_tensor(Y).cuda(eng.device), torch.as_tensor(M).cuda(eng.device), want_X=True)
        assert "scal" not in out and eng.status() == -1 and eng.launch_info()["kernel"] == KNAME[kernel]
        Xs.append(out["X"].cpu().numpy())
        eng.close()
    assert np.array_equal(Xs[0], Xs[1])


def test_want_loglik_needs_the_flag():
    from rpsmf_b200 import FilterEngine
    torch = _torch()
    eng = FilterEngine(64, 4)
    with pytest.raises(ValueError, match="loglik"):
        eng.run(torch.zeros((2, 64), dtype=torch.float64, device=eng.device), want_loglik=True)
    eng.close()


@pytest.mark.parametrize("r", [5, 16])
def test_loglik_external_exchange_matches_in_kernel(r):
    """PSMF_XCHG_EXTERNAL, one step per call (pass, caller's all-reduce -- the identity on one GPU -- then the update):
    the records match the in-kernel exchange to 1e-12."""
    torch = _torch()
    d = FLAG_D
    Y, M, C0, x0 = _masked(d, r, None, seed=1700 + r)
    init = impute_init(r)
    ref = _run(d, r, Y, M, C0, x0, init, robust=True, ll_student=True, kernel=1, ctas=3, chunks=[0, T])
    eng = _engine(d, r, init, C0, x0, robust=True, ll_student=True, exchange="external", kernel=1, ctas=3)
    Yd, Md = torch.as_tensor(Y).cuda(eng.device), torch.as_tensor(M).cuda(eng.device)
    got = np.zeros((T, 10))
    for t in range(T):
        out = eng.run_split(Yd[t:t + 1], Md[t:t + 1], 1 + t, lambda buf: None, want_loglik=True)
        got[t] = out["scal"].cpu().numpy().reshape(10)
    assert eng.status() == -1
    eng.close()
    assert relerr(got[:, 8], ref["scal"][:, 8]) < 1e-12 and relerr(got[:, 9], ref["scal"][:, 9]) < 1e-12


# ---- class surface ------------------------------------------------------------------------------------------------------
def _ydict(A):
    return {k + 1: A[k].reshape(-1, 1) for k in range(A.shape[0])}


def _collect(o):
    """Wrap the class's engine.run: every call's per-step nll and log p."""
    eng = o._get_engine()
    got = []
    run = eng.run

    def wrapped(*a, **k):
        out = run(*a, **k)
        got.append((out["nll"].cpu().numpy().reshape(-1).copy(), out["logpred"].cpu().numpy().reshape(-1).copy()))
        return out
    eng.run = wrapped
    return got


def _make(kind, fn, theta0, C0, x0, T_):
    from rpsmf_b200 import PSMFIter, PSMFRecursive, rPSMFIter, rPSMFIterMissing, rPSMFRecursive
    d, r = C0.shape
    Q, R = 0.05 * np.eye(r), 2.0 * np.eye(d)
    args = (theta0.copy(), C0, 0.5 * np.eye(r), x0.reshape(r, 1), np.eye(r))
    if kind in ("rpsmf", "rpsmf_missing", "rpsmf_recursive"):
        cls = {"rpsmf": rPSMFIter, "rpsmf_missing": rPSMFIterMissing, "rpsmf_recursive": rPSMFRecursive}[kind]
        return cls(*args, Q, R, 1.8, fn, loglik=True)
    cls = PSMFRecursive if kind == "psmf_recursive" else PSMFIter
    return cls(*args, {k: Q for k in range(T_ + 1)}, {k: R for k in range(T_ + 1)}, fn, loglik=True)


def _affine_fn(r):
    def f(theta, x, t):
        th = theta.reshape(-1)
        return (0.85 * np.eye(r) + 0.1 * np.diag(np.sin(th))) @ x + (0.2 * th * th).reshape(r, 1)
    return f


CLASS_CASES = [("psmf", "walk", None), ("rpsmf", "walk", None), ("rpsmf_missing", "walk", None), ("psmf", "external", None),
               ("psmf_recursive", "walk", 1), ("psmf_recursive", "walk", 7), ("rpsmf_recursive", "walk", 7),
               ("rpsmf_recursive", "external", 7)]


@pytest.mark.parametrize("kind,dyn,ue", CLASS_CASES, ids=["%s-%s-ue%s" % c for c in CLASS_CASES])
def test_classes_sum_the_engine_records(kind, dyn, ue):
    from rpsmf_b200.nonlinearities import RandomWalk
    d, r, T_, n_iter = 40, 3, 20, 3
    Y, M, C0, x0 = make_problem(d, r, T_, seed=1800, missing=0.2 if kind == "rpsmf_missing" else 0.0)
    theta0 = 0.3 + 0.1 * np.arange(r).reshape(r, 1)
    fn = RandomWalk() if dyn == "walk" else _affine_fn(r)
    o = _make(kind, fn, theta0, C0, x0, T_)
    got = _collect(o)
    y = _ydict(Y)
    if ue is not None:
        o.run(y, T_, 3, update_every=ue)
        sweeps = {1: got}
        assert len(got) == (T_ if dyn == "external" else -(-T_ // ue))
    else:
        o.optim_init()
        sweeps = {}
        for i in range(1, n_iter + 1):
            n0 = len(got)
            if kind == "rpsmf_missing":
                o.step(y, _ydict(M), i, T_)
            else:
                o.step(y, i, T_)
            sweeps[i] = got[n0:]
            o.predict(i, T_, 2)
            o.optim_update(i)
    for i, calls in sweeps.items():
        nll = np.concatenate([c[0] for c in calls])
        lp = np.concatenate([c[1] for c in calls])
        assert nll.size == T_ and np.all(nll != 0.0)
        assert abs(o._objective[i] - nll.sum()) <= 1e-12 * abs(nll.sum())
        assert abs(o._logpred[i] - lp.sum()) <= 1e-12 * abs(lp.sum())
    o.close()


def test_class_objective_against_oracle():
    """Sweep 1 of PSMFIter / rPSMFIter (random walk) against the restatement on the oracle's trajectory."""
    from rpsmf_b200.nonlinearities import RandomWalk
    d, r, T_ = 40, 3, 20
    Y, _, C0, x0 = make_problem(d, r, T_, seed=1900, missing=0.0)
    for kind, robust in (("psmf", False), ("rpsmf", True)):
        o = _make(kind, RandomWalk(), np.zeros((r, 1)), C0, x0, T_)
        o.optim_init()
        o.step(_ydict(Y), 1, T_)
        init = dict(V=0.5 * np.eye(r), P=np.eye(r), Q=0.05 * np.eye(r), rho=2.0, lam=1.8 if robust else 0.0)
        nll, lp = _reference(Y, None, C0, x0, init, robust, robust)
        assert abs(o._objective[1] - nll.sum()) <= TOL * abs(nll.sum())
        assert abs(o._logpred[1] - lp.sum()) <= TOL * abs(lp.sum())
        o.close()


def test_row_sharded_ranks_share_one_gpu():
    """Two row-sharded ranks on cuda:0 (the same-device mechanism of tests/multi_gpu_check.py): the per-step records are
    bit-identical on both ranks and within 1e-9 of the one-GPU engine, on the direct-load and the TMA-staged kernel."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29523", os.path.join(root, "tests", "multi_gpu_loglik_check.py"), "--same-device"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, PSMF_SPIN_TIMEOUT_MS="60000"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" OK") == 4 and "FAIL" not in r.stdout
