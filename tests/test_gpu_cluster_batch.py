"""Batched engines of large series: one thread-block cluster of CTAs per series.

An engine of several series gives each series a cluster of `ctas` CTAs (2..16) when asked to, or when one CTA per series
no longer holds a series.  The CTAs of a cluster sum their statistics through distributed shared memory with the 16-wide
addition tree of the cooperative single-series path, so a cluster of c CTAs gives the bits of a single-series engine
created with kernel=1, ctas=c.  Most cases here check exactly that, bit for bit, over two launches; the others check the
automatic size against the float64 oracle, the waves of clusters that do not all fit the device, the shapes that keep
their kernel, the refusals and the tools at the new sizes.  Every case checks through launch_info() that the variant
it is about ran: the direct-load kernel with the intended number of CTAs per series.
"""

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _compare, _oracle_run

pytestmark = pytest.mark.gpu

TOL32 = 1e-4
RANKS = list(range(1, 17))
SPLIT_RANKS = [5, 8, 9, 16]
T = 12
CHUNKS = [0, 5, 12]                # two launches: the pending rank-1 update is flushed at the launch boundary
D_BIT = 4001                       # 126 tiles; the last tile holds one row


def _torch():
    import torch
    return torch


def _dtype(tag):
    torch = _torch()
    return torch.float64 if tag == "f64" else torch.float32


def _rounded(a, tag):
    return a if tag == "f64" else a.astype(np.float32).astype(np.float64)


def _init(r, d=None, rho_vector=False, seed=0):
    init = impute_init(r)
    if rho_vector:
        init["rho"] = 10.0 * (0.5 + np.random.RandomState(seed).rand(d))
    return init


def _engine(d, r, S, init, C0, x0, theta=None, A=None, c=None, **kw):
    from rpsmf_b200 import FilterEngine
    eng = FilterEngine(d, r, n_series=S, **kw)
    rho = init["rho"]
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=rho if np.ndim(rho) else [rho], lam=[init["lam"]],
                  theta=theta)
    if A is not None:
        eng.set_linear_dynamics(A, c)
    return eng


def _run(d, r, Y, M, C0, x0, init, S, chunks=CHUNKS, tag="f64", want_grad=False, E=None, Yorig=None, theta=None, A=None, c=None,
         ext=None, **kw):
    """Filter Y (S, T, d) on one engine of S series in the launches of `chunks`.  `ext` = (xbar (S, T, r), F (S, T, r, r)): external
    dynamics, one step per launch.  Returns a dict of host arrays with the series axis first, and launch_info."""
    torch = _torch()
    dt = _dtype(tag)
    eng = _engine(d, r, S, init, C0, x0, theta=theta, A=A, c=c, dtype=dt, **kw)
    dev = eng.device
    Yd = torch.as_tensor(Y).to(dev, dt)
    Md = None if M is None else torch.as_tensor(M).to(dev)
    Ed = None if E is None else torch.as_tensor(E).to(dev)
    Yod = None if Yorig is None else torch.as_tensor(Yorig).to(dev, dt)
    if ext is not None:
        chunks = list(range(Y.shape[1] + 1))
    acc = dict(X=[], Yrec=[], scal=[])
    grad, ev = None, None
    for a, b in zip(chunks[:-1], chunks[1:]):
        xkw = {} if ext is None else dict(xbar=ext[0][:, a], F=ext[1][:, a])
        out = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, want_Yrec=True, want_scal=True,
                      want_grad=want_grad, E=None if Ed is None else Ed[:, a:b], Yorig=None if Yod is None else Yod[:, a:b], **xkw)
        assert eng.status() == -1
        sq = (lambda v: v.unsqueeze(0)) if S == 1 else (lambda v: v)
        acc["X"].append(sq(out["X"]).cpu().numpy())
        acc["Yrec"].append(sq(out["Yrec"]).double().cpu().numpy())
        acc["scal"].append(sq(out["scal"]).cpu().numpy())
        if want_grad:
            g = np.concatenate([sq(out["grad_A"]).reshape(S, -1).cpu().numpy(), sq(out["grad_c"]).cpu().numpy()], axis=1) \
                if "grad_A" in out else sq(out["grad"]).cpu().numpy()
            grad = g if grad is None else grad + g
        if E is not None:
            e = sq(out["eval"]).cpu().numpy()
            ev = e if ev is None else ev + e
    res = {k: np.concatenate(v, axis=1) for k, v in acc.items()}
    st = eng.get_state()
    for k, v in st.items():
        v = v.unsqueeze(0) if S == 1 else v
        res[k] = v.double().cpu().numpy()
    res["grad"], res["eval"], res["info"] = grad, ev, eng.launch_info()
    eng.close()
    return res


KEYS = ("X", "Yrec", "scal", "C", "P", "V", "Q", "x", "rho", "lam", "grad", "eval")


def _bits_equal(a, b, s=None):
    """a (one engine of S series) against b (series s of a single-series run, or a whole batched run when s is None)."""
    for k in KEYS:
        if a[k] is None:
            assert b[k] is None, k
            continue
        va = a[k] if s is None else a[k][s:s + 1]
        assert va.shape == b[k].shape, (k, va.shape, b[k].shape)
        assert np.array_equal(va, b[k]), (k, float(np.max(np.abs(va - b[k]))))


def _check_cluster(info, c):
    assert info["kernel"] == "direct" and info["ctas"] == c and info["threads"] == 256, info


def _vs_single(d, r, Y, M, C0, x0, init, S, ncta, tag="f64", **kw):
    """The engine of S series with clusters of ncta CTAs against S single-series cooperative engines with ctas = ncta, bit
    for bit."""
    res = _run(d, r, Y, M, C0, x0, init, S, tag=tag, ctas=ncta, kernel=1, **kw)
    _check_cluster(res["info"], ncta)
    for s in range(S):
        one = {k: v for k, v in kw.items() if k not in ("theta", "E", "Yorig", "ext")}
        sel = lambda a: None if a is None else a[s:s + 1]
        ext = kw.get("ext")
        rho = init["rho"]
        init_s = dict(init, rho=rho[s] if np.ndim(rho) > 1 else rho)
        ref = _run(d, r, Y[s:s + 1], sel(M), C0[s], x0[s], init_s, 1, tag=tag, ctas=ncta, kernel=1, theta=sel(kw.get("theta")),
                   E=sel(kw.get("E")), Yorig=sel(kw.get("Yorig")), ext=None if ext is None else (sel(ext[0]), sel(ext[1])), **one)
        info = ref["info"]
        assert info["kernel"] == "direct" and info["ctas"] == ncta, info
        _bits_equal(res, ref, s)
    return res


def _masked(d, r, S, seed, dead=True):
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, S=S)
    rows = np.array([1, d // 2, d - 1])
    if dead:
        M[..., rows] = 0
        Y = Y * M
    return Y, M, C0, x0, rows


# ---- 1. bit-identity with the cooperative single-series path -----------------------------------------------------------
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", RANKS)
def test_cluster_bits_equal_cooperative_single_series(r, tag):
    Y, M, C0, x0, _ = _masked(D_BIT, r, 3, seed=r)
    _vs_single(D_BIT, r, _rounded(Y, tag), M, _rounded(C0, tag), x0, _init(r), 3, 3, tag=tag, robust=True)


# ---- 2. the automatic size just past the one-CTA limit, against the float64 oracle --------------------------------------
_LIMIT = {}


def _one_cta_limit(r, tag):
    """Smallest whole-tile row count at which an engine of 2 series no longer runs one CTA per series (binary search over
    engine creation; launch_info of a run is checked by the callers)."""
    key = (r, tag)
    if key in _LIMIT:
        return _LIMIT[key]
    from rpsmf_b200 import FilterEngine

    def cluster(nt):
        eng = FilterEngine(32 * nt, r, n_series=2, dtype=_dtype(tag), kernel=1)
        try:
            return eng._h is not None and _plan_ctas(eng) > 1
        finally:
            eng.close()
    lo, hi = 32, 4096
    assert not cluster(lo) and cluster(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if cluster(mid):
            hi = mid
        else:
            lo = mid
    _LIMIT[key] = 32 * hi
    return _LIMIT[key]


def _plan_ctas(eng):
    """CTAs per series the engine plans (a one-step run of zeros reports it)."""
    torch = _torch()
    Y = torch.zeros((eng.S, 1, eng.d), dtype=eng.dtype, device=eng.device)
    eng.run(Y, None, want_X=False)
    eng.status()
    return eng.launch_info()["ctas"]


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", RANKS)
def test_auto_size_past_the_one_cta_limit_against_oracle(r, tag):
    d = _one_cta_limit(r, tag) + 7                 # a partial last tile
    S = 3
    Y, M, C0, x0, dead = _masked(d, r, S, seed=100 + r)
    Y, C0 = _rounded(Y, tag), _rounded(C0, tag)
    init = _init(r)
    res = _run(d, r, Y, M, C0, x0, init, S, tag=tag, robust=True)
    info = res["info"]
    assert info["kernel"] == "direct" and 2 <= info["ctas"] <= 16, info
    tol = TOL if tag == "f64" else TOL32
    for s in range(S):
        ref = _oracle_run(Y[s], M[s], C0[s], x0[s], init, po.OracleConfig(robust=True))
        got = (res["X"][s], res["Yrec"][s], res["scal"][s], {k: res[k][s] for k in ("C", "P", "V", "Q", "x", "rho", "lam")}, info)
        _compare(got, ref, tol)
        # rows never observed keep C bit for bit
        assert np.array_equal(res["C"][s][dead], C0[s][dead].astype(np.float32 if tag == "f32" else np.float64).astype(np.float64))
    if r == 1:
        # a step with every row missing stays finite (x'Vx vanishes after it at r = 1; the reference gives NaN there): a pure
        # prediction step
        M[:, 6] = 0
        res = _run(d, r, Y * M, M, C0, x0, init, S, tag=tag, robust=True)
        assert info["ctas"] == res["info"]["ctas"]
        assert np.isfinite(res["X"]).all() and np.isfinite(res["C"]).all() and np.isfinite(res["V"]).all()
        assert np.array_equal(res["X"][:, 6], res["X"][:, 5])


# ---- 3. flags: bit-identical to the single-series cooperative engines, and against the oracle ------------------------------
FLAG_CASES = ["psmf_vt", "psmf_v", "fixed_lambda", "alpha_beta", "simplified_cos", "rho_vector", "loglik", "grad_linear",
              "external", "eval"]


def _flag_setup(case, d, r, S, seed):
    """(engine keywords, run keywords, init, oracle config or None)."""
    rng = np.random.RandomState(seed)
    init = _init(r)
    cfg = None
    kw, rk = dict(robust=True), {}
    if case == "psmf_vt":
        kw, cfg = dict(robust=False, c_update_transpose=True), po.OracleConfig(robust=False, c_update_transpose=True)
        init["lam"] = 0.0
    elif case == "psmf_v":
        kw, cfg = dict(robust=False, c_update_transpose=False), po.OracleConfig(robust=False, c_update_transpose=False)
        init["lam"] = 0.0
    elif case == "fixed_lambda":
        kw["fixed_lambda"], cfg = True, po.OracleConfig(robust=True, fixed_lambda=True)
    elif case == "alpha_beta":
        kw.update(alpha=0.97, beta=1.03)
        cfg = po.OracleConfig(robust=True, alpha=0.97, beta=1.03)
    elif case == "simplified_cos":
        kw.update(simplified=True, dynamics=1)
        rk.update(theta=0.01 * rng.rand(S, r), want_grad=True)
    elif case == "rho_vector":
        kw["rho_vector"] = True
        init["rho"] = np.stack([_init(r, d, True, seed + s)["rho"] for s in range(S)])
    elif case == "loglik":
        kw.update(loglik=True)
    elif case == "grad_linear":
        A = 0.9 * np.eye(r) + 0.02 * rng.randn(r, r)
        c = 0.05 * rng.randn(r)
        kw.update(dynamics=2, grad_linear=True, loglik=(seed % 2 == 0))
        rk.update(A=A, c=c, want_grad=True)
        cfg = po.OracleConfig(robust=True, dynamics=po.DYN_LINEAR, lin_A=A, lin_c=c)
    elif case == "external":
        xb = rng.rand(S, T, r)
        F = 0.9 * np.eye(r) + 0.01 * rng.randn(S, T, r, r)
        kw.update(dynamics=3)
        rk.update(ext=(xb, F), want_grad=True)
    return kw, rk, init, cfg


@pytest.mark.parametrize("case", FLAG_CASES)
@pytest.mark.parametrize("r", SPLIT_RANKS)
def test_flags_bit_identical_to_single_series(r, case):
    S, c, d = 3, 3, D_BIT
    Y, M, C0, x0, _ = _masked(d, r, S, seed=200 + r)
    kw, rk, init, cfg = _flag_setup(case, d, r, S, seed=r)
    if case == "eval":
        rng = np.random.RandomState(r)
        E = (rng.rand(S, T, d) < 0.15).astype(np.uint8)
        rk.update(E=E, Yorig=Y + 0.1 * rng.randn(S, T, d))
    res = _vs_single(d, r, Y, M, C0, x0, init, S, c, **kw, **rk)
    if case == "loglik":
        assert res["scal"].shape[-1] == 10 and np.isfinite(res["scal"][..., 8:]).all()
    else:
        assert res["scal"].shape[-1] == (10 if kw.get("loglik") else 8)      # a plain run through the cluster variant: 8 wide
    if case == "eval":
        E = rk["E"]
        assert np.array_equal(res["eval"][:, 2], E.reshape(S, -1).sum(axis=1).astype(np.float64))
    if cfg is not None:
        for s in range(S):
            ref = _oracle_run(Y[s], M[s], C0[s], x0[s], init, cfg)
            got = (res["X"][s], res["Yrec"][s], res["scal"][s], {k: res[k][s] for k in ("C", "P", "V", "Q", "x", "rho", "lam")}, None)
            _compare(got, ref, TOL)


@pytest.mark.parametrize("r", SPLIT_RANKS)
def test_nan_mask_same_bits_as_byte_mask(r):
    S, c, d = 3, 3, D_BIT
    Y, M, C0, x0, _ = _masked(d, r, S, seed=300 + r)
    init = _init(r)
    byte = _run(d, r, Y, M, C0, x0, init, S, ctas=c, kernel=1, robust=True)
    Yn = np.where(M != 0, Y, np.nan)
    nan = _run(d, r, Yn, None, C0, x0, init, S, ctas=c, kernel=1, robust=True, nan_mask=True)
    _check_cluster(byte["info"], c)
    _check_cluster(nan["info"], c)
    _bits_equal(nan, byte)


# ---- 4. cluster sizes and waves of clusters -----------------------------------------------------------------------------
@pytest.mark.parametrize("c", [2, 3, 5, 8, 16])
@pytest.mark.parametrize("r", [1, 16])
def test_cluster_sizes(r, c):
    S = 3
    Y, M, C0, x0, _ = _masked(D_BIT, r, S, seed=400 + c)
    _vs_single(D_BIT, r, Y, M, C0, x0, _init(r), S, c, robust=True)


def test_clusters_in_waves_against_oracle_and_status():
    """S * c above what the device holds at once: the clusters run in waves.  An inf planted in one series is reported."""
    torch = _torch()
    S, c, r, d = 40, 16, 8, 6000
    Y, M, C0, x0, _ = _masked(d, r, S, seed=5)
    init = _init(r)
    res = _run(d, r, Y, M, C0, x0, init, S, ctas=c, kernel=1, robust=True)
    _check_cluster(res["info"], c)
    assert S * c > torch.cuda.get_device_properties(0).multi_processor_count * 2
    for s in range(S):
        ref = _oracle_run(Y[s], M[s], C0[s], x0[s], init, po.OracleConfig(robust=True))
        got = (res["X"][s], res["Yrec"][s], res["scal"][s], {k: res[k][s] for k in ("C", "P", "V", "Q", "x", "rho", "lam")}, None)
        _compare(got, ref, TOL)
    # a planted inf in series 17 at step 4: the status word names the first bad step, as in a batched engine of one CTA per series
    Yb = Y.copy()
    Yb[17, 4, 10] = np.inf
    Mb = M.copy()
    Mb[17, 4, 10] = 1
    eng = _engine(d, r, S, init, C0, x0, robust=True, ctas=c, kernel=1)
    eng.run(torch.as_tensor(Yb).cuda(), torch.as_tensor(Mb).cuda(), want_X=True)
    assert eng.status() == 4
    _check_cluster(eng.launch_info(), c)
    eng.close()


# ---- 5. shapes that run today keep their kernel ------------------------------------------------------------------------------
@pytest.mark.parametrize("name,kernel,d,want", [("direct_S3", 1, 4001, ("direct", 1, 256)), ("batch8", 3, 1100, ("batch", 1, 256)),
                                                ("batch4", 3, 203, ("batch", 1, 128))])
def test_shapes_of_today_keep_their_kernel(name, kernel, d, want):
    r, S = 8, 3
    Y, M, C0, x0, _ = _masked(d, r, S, seed=6, dead=False)
    init = _init(r)
    res = _run(d, r, Y, M, C0, x0, init, S, kernel=kernel, robust=True)
    info = res["info"]
    assert (info["kernel"], info["ctas"], info["threads"]) == want, info
    ref = _oracle_run(Y[1], M[1], C0[1], x0[1], init, po.OracleConfig(robust=True))
    assert relerr(res["X"][1], ref[1]) < TOL


# ---- 6. refusals ----------------------------------------------------------------------------------------------------------------
def test_refusals_and_a_fresh_engine_after_them():
    from rpsmf_b200 import FilterEngine
    from rpsmf_b200._capi import PsmfError
    with pytest.raises(PsmfError, match="cluster size of a series, 1..16"):
        FilterEngine(D_BIT, 8, n_series=3, ctas=17)
    # a series so long that even 16 CTAs cannot hold its residuals: the message names the row limit
    with pytest.raises(PsmfError, match=r"d too large for a batched engine.*rows at r = 16"):
        FilterEngine(1_000_000, 16, n_series=2)
    # a forced cluster too small for the series
    with pytest.raises(PsmfError, match="cannot schedule a cluster of 2 CTAs"):
        FilterEngine(200_000, 16, n_series=2, ctas=2)
    # a run refused for its shared memory (evaluation buffers behind a nearly full residual buffer) leaves the engine as it
    # was: the next run gives the bits of a fresh engine.  The shape: a little under the row limit the refusal above names.
    import re
    torch = _torch()
    r, S = 16, 2
    try:
        FilterEngine(1_000_000, r, n_series=S)
    except PsmfError as e:
        m = re.search(r"at most (\d+) CTAs here, which holds about (\d+) rows", str(e))
    c, d = int(m.group(1)), int(m.group(2)) - 100
    Y, M, C0, x0, _ = _masked(d, r, S, seed=7, dead=False)
    init = _init(r)
    eng = _engine(d, r, S, init, C0, x0, robust=True, ctas=c, kernel=1)
    E = torch.ones((S, T, d), dtype=torch.uint8, device=eng.device)
    Yd, Md = torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda()
    with pytest.raises(PsmfError, match="no shared memory left"):
        eng.run(Yd, Md, want_X=True, E=E, Yorig=Yd)
    X1 = eng.run(Yd, Md, want_X=True)["X"].cpu().numpy()
    assert eng.status() == -1
    _check_cluster(eng.launch_info(), c)
    eng.close()
    fresh = _engine(d, r, S, init, C0, x0, robust=True, ctas=c, kernel=1)
    X2 = fresh.run(Yd, Md, want_X=True)["X"].cpu().numpy()
    fresh.close()
    assert np.array_equal(X1, X2)


# ---- 7. tools at the new sizes ----------------------------------------------------------------------------------------------------
def test_eval_full_and_predict_past_the_grid_stride_caps():
    torch = _torch()
    r, S, d = 8, 3, 70_000
    Y, M, C0, x0, _ = _masked(d, r, S, seed=8, dead=False)
    init = _init(r)
    eng = _engine(d, r, S, init, C0, x0, robust=True)
    Yd, Md = torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda()
    out = eng.run(Yd, Md, want_X=True)
    assert eng.status() == -1
    info = eng.launch_info()
    assert info["kernel"] == "direct" and info["ctas"] > 1, info
    C = eng.get_state()["C"].cpu().numpy()
    X = out["X"]
    rng = np.random.RandomState(8)
    Yo = rng.randn(S, T, d)
    E = (rng.rand(S, T, d) < 0.3).astype(np.uint8)
    ef = eng.eval_full(X, torch.as_tensor(Yo).cuda(), torch.as_tensor(E).cuda()).cpu().numpy()
    Xh = X.cpu().numpy()
    for s in range(S):
        pred = Xh[s] @ C[s].T
        sq = ((pred - Yo[s]) ** 2)[E[s] != 0].sum()
        assert abs(ef[s, 0] - sq) <= 1e-12 * sq and ef[s, 1] == E[s].sum()
    Xp, Yp = eng.predict(4, T + 1)
    Xp, Yp = Xp.cpu().numpy(), Yp.cpu().numpy()
    for s in range(S):
        ref = Xp[s] @ C[s].T
        assert relerr(Yp[s], ref) < 1e-12
    eng.close()


def test_fit_repeats_at_a_size_refused_before():
    """4 repeats of the imputation experiment at a row count one CTA per series cannot hold: the batch against the
    per-repeat functions (1e-9), and its X against the float64 oracle."""
    from rpsmf_b200 import impute
    r, n, Iter, S = 16, 10, 1, 4
    d = _one_cta_limit(r, "f64") + 64
    rng = np.random.RandomState(9)
    Ct = rng.randn(d, r)
    Xt = np.cumsum(0.1 * rng.randn(r, n), axis=1)
    Yfull = Ct @ Xt + 0.3 * rng.randn(d, n)
    V, Q0, P, R0 = 2.0 * np.eye(r), 0.1 * np.eye(r), np.eye(r), 10.0
    Ys, Cs, Xs, Ms, Mm = [], [], [], [], []
    for k in range(S):
        rk = np.random.RandomState(100 + k)
        Mmiss = (rk.rand(d, n) < 0.1).astype(float)
        M = (rk.rand(d, n) >= 0.1).astype(float) * (1 - Mmiss)
        Ys.append(np.where(M != 0, Yfull, np.nan)); Cs.append(rk.rand(d, r)); Xs.append(rk.rand(r, n)); Ms.append(M); Mm.append(Mmiss)
    Ei = [1.0] * S
    Xb = [x.copy() for x in Xs]
    Ep, Ef, _, Ins = impute.fit_repeats(Ys, [c.copy() for c in Cs], Xb, Ms, Mm, V, Q0, R0, P, 1.8, 2.0, Iter, Yfull, Ei)
    info = impute.fit_repeats.last_launch
    assert info["kernel"] == "direct" and info["ctas"] > 1, info
    for k in range(S):
        Xk = Xs[k].copy()
        ep, ef, _, ins = impute.robust_PSMF(Ys[k], Cs[k].copy(), Xk, d, n, r, Ms[k], Mm[k], V, Q0, R0, P, 1.8, 2.0, Iter, Yfull, Ei[k])
        assert relerr(np.asarray(Ep[k]), np.asarray(ep)) < TOL and relerr(np.asarray(Ef[k]), np.asarray(ef)) < TOL
        assert abs(Ins[k] - ins) < 1e-12
        assert relerr(Xb[k], Xk) < TOL
        init = dict(V=V, Q=Q0, P=P, rho=10.0, lam=1.8)
        ref = _oracle_run(np.nan_to_num(Ys[k]).T.copy(), Ms[k].T.astype(np.uint8), Cs[k], Xs[k][:, n - 1].copy(), init,
                          po.OracleConfig(robust=True))
        assert relerr(Xb[k].T, ref[1]) < TOL
