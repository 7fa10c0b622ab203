"""Fused evaluation, the forecast and the data tools on every kernel variant, rank and storage type against float64
references.

The imputation experiment publishes three numbers the filter kernels do not use themselves: Epred and the sig-sigma
coverage count, accumulated inside the row pass of the direct-load and batch kernels (a row's prediction waits in
shared memory and is scored one pass later, or in the flush after the last step of a launch), and Efull from
psmf_eval_full.  The forecast (psmf_predict: roll-out and projection) and the handle-free tools (ingest, mask transpose,
the missing-segment generator, the NaN count) sit on either side of the filter.  Each case here forces its kernel and
checks through launch_info() that the variant it is about is the one that ran.

References: the pinned oracle's trajectory for the evaluation (coverage counts and entry counts exact, sums fp64 1e-9 /
fp32 1e-4), numpy float64 for eval_full and the projection (1e-12; fp32 output within one ulp of the rounded
reference), the oracle's dynamics for the roll-out (1e-12), and bit-exact numpy restatements for the tools.
"""

import ctypes as C

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import _engine_run, _oracle_run, _padded, _torch
from test_gpu_kernel_matrix import KNAME, RANKS, SPLIT_RANKS, VARIANTS, _check_variant, _dtype, _rounded, _sms

pytestmark = pytest.mark.gpu

EVAL_T = 12
EVAL_CHUNKS = [0, 1, 5, EVAL_T]     # a one-step launch, coverage scored in each flush, state carried across launches
EVAL_VARIANTS = ["direct", "direct_S3", "rhovec", "rhovec_S3", "batch8", "batch4"]
MIN_FLIPS = 3                       # entries by which a wrong interval must move the coverage count of a cell


def _stream():
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# ---- 1. fused evaluation against the oracle --------------------------------------------------------------------------
def _eval_init(r, d, rho_vector, seed):
    """V = 20 I and rho = 1 (the suite's usual start is V = 2 I, rho = 10): a = x'Vx stays a sizeable part of
    U = a m_i + eta, so the coverage count tells the a m_i term, and the step its a comes from, apart."""
    init = impute_init(r)
    init["V"] = 20.0 * np.eye(r)
    init["rho"] = 0.5 + np.random.RandomState(seed).rand(d) if rho_vector else 1.0
    return init


def _direct_cps(d):
    """CTAs of an automatic direct-load grid for one series (psmf_create): ntiles / 16, at most one per SM."""
    return max(1, min((d + 31) // 32 // 16, _sms()))


def _eval_marks(M, cps, dead, rng):
    """E over (T, d): about 15 % of the entries, half on observed and half on missing ones, plus every step of row d - 1
    (the partial last tile), of the rows either side of each CTA boundary and of the never-observed row `dead`."""
    T, d = M.shape
    obs = M == 1
    u = rng.rand(T, d)
    E = (obs & (u < 0.075 / obs.mean())) | (~obs & (u < 0.075 / (~obs).mean()))
    ntiles = (d + 31) // 32
    rows = [d - 1, dead] + [32 * (ntiles * p // cps) + o for p in range(1, cps) for o in (-1, 0)]
    E[:, rows] = True
    return E.astype(np.uint8)


def _coverage_reference(Y, M, C0, x0, init, cfg, E, tag, rng):
    """One series.  Yorig is built on the oracle's trajectory, which does not depend on it: yhat + u h with h the half-width
    of the interval and u uniform in [-2, 2] without 0.98 <= |u| <= 1.02, so that no value lies within 2 % of h of a bound
    (the count is exact under fp32 drift), rounded to fp32 for fp32 storage, NaN where E = 0 (never read).  Returns the
    oracle result, Yorig, the sum of squared errors, the coverage count, and the counts with U = eta and with the a of
    step t + 1 (what the kernels would report if they dropped the a m_i term or read a from the wrong step)."""
    rec = []
    ref = _oracle_run(Y, M, C0, x0, init, cfg, record=rec)
    yhat = np.stack([o["yhat"] for o in rec])
    lo, hi = np.stack([o["lo"] for o in rec]), np.stack([o["hi"] for o in rec])
    h = 0.5 * (hi - lo)
    u = rng.uniform(-2.0, 2.0, yhat.shape)
    while True:
        bad = np.abs(np.abs(u) - 1.0) <= 0.02
        if not bad.any():
            break
        u[bad] = rng.uniform(-2.0, 2.0, int(bad.sum()))
    Yo = _rounded(yhat + u * h, tag)
    Yo[E == 0] = np.nan
    sel = E == 1
    sse = float(np.sum((yhat[sel] - Yo[sel]) ** 2))

    def inside(lo_, hi_):
        return int(np.sum((Yo[sel] < hi_[sel]) & (lo_[sel] < Yo[sel])))

    count = inside(lo, hi)
    eta = np.array([o["eta"] for o in rec])[:, None]
    a = np.array([o["a"] for o in rec])
    ost = ref[0]
    a_next = np.append(a[1:], ost.x @ ost.V @ ost.x)[:, None]       # identity dynamics: x_bar of step t + 1 is x_t
    m = M.astype(float)
    alt = []
    for U in (eta + 0.0 * m, a_next * m + eta):
        s = cfg.sig * np.sqrt(U)
        alt.append(inside(yhat - s, yhat + s))
    return ref, Yo, sse, count, alt


def _eval_problem(d, r, S, tag, robust, sig, cps, rho_vector, seed, T=EVAL_T):
    """A masked problem with a never-observed row, the start of _eval_init, E and Yorig per series, and the references."""
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, S=S)
    dead = d // 2
    M[..., dead] = 0
    Y = Y * M
    init = _eval_init(r, d, rho_vector, seed)
    cfg = po.OracleConfig(robust=robust, c_update_transpose=robust, bounds_rpsmf=robust, sig=sig)
    rng = np.random.RandomState(seed + 1)
    refs, Es, Yos = [], [], []
    for s in range(S or 1):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        E = _eval_marks(one(M), cps, dead, rng)
        ref, Yo, sse, count, alt = _coverage_reference(_rounded(one(Y), tag), one(M), _rounded(one(C0), tag), one(x0), init,
                                                       cfg, E, tag, rng)
        refs.append((ref, sse, count, alt))
        Es.append(E)
        Yos.append(Yo)
    E, Yorig = (Es[0], Yos[0]) if S is None else (np.stack(Es), np.stack(Yos))
    return Y, M, C0, x0, init, E, Yorig, refs


def _check_eval(res, E, refs, S, tag, sensitive):
    """Per series: the entry count and the coverage count exactly, the squared error to the storage type's tolerance,
    entry 3 zero, X and C against the oracle; and with `sensitive`, on the reference side, that the data tell a wrong U
    (the a m_i term dropped, or a taken from step t + 1) apart from the right one."""
    from rpsmf_b200 import _capi
    tol = _dtype(tag)[2]
    X, _, _, st, _ = res
    ev = np.atleast_2d(st["eval"])
    flips = np.zeros(2)
    for s, (ref, sse, count, alt) in enumerate(refs):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        ost, oX, _, _ = ref
        assert ev[s, _capi.EVAL_COUNT] == float(one(E).sum()), s
        assert ev[s, _capi.EVAL_INSIDE] == float(count), (s, ev[s], count)
        assert abs(ev[s, _capi.EVAL_SSE] - sse) <= tol * sse, (s, ev[s], sse)
        assert ev[s, 3] == 0.0
        assert relerr(one(X), oX) < tol and relerr(one(st["C"]), ost.C) < tol, s
        flips += np.abs(count - np.array(alt))
    if sensitive:
        assert (flips >= MIN_FLIPS).all(), flips


EVAL_PARAMS = [(n, r, t, True) for n in EVAL_VARIANTS for r in RANKS for t in ("f64", "f32")] + \
              [(n, r, t, False) for n in EVAL_VARIANTS for r in SPLIT_RANKS for t in ("f64", "f32")]


@pytest.mark.parametrize("name,r,tag,robust", EVAL_PARAMS,
                         ids=["%s-%s-r%d-%s" % ("rpsmf" if b else "psmf", n, r, t) for n, r, t, b in EVAL_PARAMS])
def test_fused_evaluation_matrix(name, r, tag, robust):
    kernel, d, S, kw = VARIANTS[name]
    dtype, esize, _ = _dtype(tag)
    sig = 1.5 if r % 4 == 3 else 2.0
    cps = _direct_cps(d) if kernel == 1 and S is None else 1
    Y, M, C0, x0, init, E, Yorig, refs = _eval_problem(d, r, S, tag, robust, sig, cps, kw.get("rho_vector", False),
                                                       seed=1000 + 37 * r + d % 89)
    res = _engine_run(d, r, Y, M, C0, x0, init, robust, dtype=dtype, chunks=EVAL_CHUNKS, S=S, kernel=kernel,
                      c_update_transpose=robust, Yorig=Yorig, E=E, sig=sig, **kw)
    _check_variant(name, res[4], r, esize, d)
    assert res[4]["ctas"] == cps and res[4]["launches"] == 2, res[4]
    _check_eval(res, E, refs, S, tag, robust)


# ---- 2. evaluation composed with the log-likelihood and the linear-dynamics gradient ---------------------------------
def _composed_run(d, r, S, kernel, prob, E=None, Yorig=None, nan_mask=False, **flags):
    """Linear dynamics over EVAL_CHUNKS; returns every output per launch and the final state, as numpy arrays."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    Y, M, C0, x0, init, A, c = prob
    eng = FilterEngine(d, r, n_series=S, kernel=kernel, dynamics=_capi.DYN_LINEAR, nan_mask=nan_mask, **flags)
    eng.set_linear_dynamics(A, c)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    dev = eng.device
    Yd = torch.as_tensor(np.where(M == 1, Y, np.nan) if nan_mask else Y).to(dev)
    Md = None if nan_mask else torch.as_tensor(M).to(dev)
    Yod = None if E is None else torch.as_tensor(Yorig).to(dev)
    Ed = None if E is None else torch.as_tensor(E).to(dev)
    out = {}
    for a, b in zip(EVAL_CHUNKS[:-1], EVAL_CHUNKS[1:]):
        o = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, want_scal=True,
                    want_grad=flags.get("grad_linear", False), Yorig=None if E is None else Yod[:, a:b],
                    E=None if E is None else Ed[:, a:b])
        assert eng.status() == -1
        for k, v in o.items():
            out.setdefault(k, []).append(v.cpu().numpy())
    out["state"] = {k: v.cpu().numpy() for k, v in eng.get_state().items()}
    out["info"] = eng.launch_info()
    eng.close()
    return out


def _same(a, b, keys):
    for k in keys:
        for x, y in zip(a[k], b[k]):
            assert np.array_equal(x, y, equal_nan=True), k


COMPOSED = [(1, 4001, 1), (3, 1100, 3)]


@pytest.mark.parametrize("kernel,d,S", COMPOSED, ids=[KNAME[k] for k, _, _ in COMPOSED])
@pytest.mark.parametrize("r", [5, 16])
def test_evaluation_composed_with_loglik_and_linear_gradient(kernel, d, S, r):
    """The gradient accumulator G_A sits behind the evaluation buffers (glin_off): the evaluation record must not
    depend on the other variants, and nothing else may depend on the evaluation."""
    Y, M, C0, x0 = make_problem(d, r, EVAL_T, seed=300 + r, S=S)
    rng = np.random.RandomState(r)
    A = 0.9 * np.eye(r) + 0.05 * rng.randn(r, r) / np.sqrt(r)
    c = 0.1 * rng.randn(r)
    init = impute_init(r)
    prob = (Y, M, C0, x0, init, A, c)
    cps = _direct_cps(d) if kernel == 1 else 1
    E = np.stack([_eval_marks(M[s], cps, d // 2, rng) for s in range(S)])
    Yorig = np.where(E == 1, Y + rng.randn(*Y.shape), np.nan)
    every = dict(loglik=True, grad_linear=True)
    full = _composed_run(d, r, S, kernel, prob, E, Yorig, **every)
    assert full["info"]["kernel"] == KNAME[kernel] and full["info"]["ctas"] == cps, full["info"]
    no_eval = _composed_run(d, r, S, kernel, prob, **every)
    _same(full, no_eval, ("X", "scal", "grad_A", "grad_c"))
    for k in ("C", "V", "P", "x", "Q", "rho", "lam"):
        assert np.array_equal(full["state"][k], no_eval["state"][k]), k
    plain = _composed_run(d, r, S, kernel, prob, E, Yorig)
    assert plain["info"]["kernel"] == KNAME[kernel]
    _same(full, plain, ("eval", "X"))
    nan = _composed_run(d, r, S, kernel, prob, E, Yorig, nan_mask=True, **every)
    _same(full, nan, ("eval", "X", "grad_A", "grad_c"))
    assert sum(float(np.sum(e[..., 2])) for e in full["eval"]) == E.sum()


# ---- 3. dispatch and refusal with evaluation -------------------------------------------------------------------------
def test_batch_fallback_when_evaluation_buffers_do_not_fit():
    """S = 2, r = 16, fp32, d = 2600 (82 tiles): the batch kernel holds C and the residuals (188 928 bytes) but not the
    evaluation buffers as well (233 552 bytes, over the 232 448-byte opt-in limit).  Automatic dispatch falls back to
    the direct-load kernel and matches the oracle; forcing the batch kernel raises, after which the engine still gives
    the bits of a fresh one."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r, S, tag = 2600, 16, 2, "f32"
    dtype = _dtype(tag)[0]
    Y, M, C0, x0, init, E, Yorig, refs = _eval_problem(d, r, S, tag, True, 2.0, 1, False, seed=2600)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, dtype=dtype, chunks=EVAL_CHUNKS, S=S)
    assert res[4]["kernel"] == "batch", res[4]
    res = _engine_run(d, r, Y, M, C0, x0, init, True, dtype=dtype, chunks=EVAL_CHUNKS, S=S, Yorig=Yorig, E=E)
    assert res[4]["kernel"] == "direct", res[4]
    _check_eval(res, E, refs, S, tag, True)

    def fresh(eng=None):
        if eng is None:
            eng = FilterEngine(d, r, n_series=S, dtype=dtype, kernel=3)
        eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        out = eng.run(torch.as_tensor(Y).to(dtype).cuda(), torch.as_tensor(M).cuda(), want_X=True)
        assert eng.status() == -1 and eng.launch_info()["kernel"] == "batch"
        return out["X"].cpu().numpy(), eng.get_state()["C"].cpu().numpy()

    Xa, Ca = fresh()
    eng = FilterEngine(d, r, n_series=S, dtype=dtype, kernel=3)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd = torch.as_tensor(Y).to(dtype).cuda()
    with pytest.raises(_capi.PsmfError):
        eng.run(Yd, torch.as_tensor(M).cuda(), Yorig=torch.as_tensor(Yorig).to(dtype).cuda(), E=torch.as_tensor(E).cuda())
    Xb, Cb = fresh(eng)
    assert np.array_equal(Xa, Xb) and np.array_equal(Ca, Cb)
    eng.close()


@pytest.mark.parametrize("case", ["tma", "external"])
def test_evaluation_refused(case):
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r = 960, 8
    Y, M, C0, x0 = make_problem(d, r, 4, seed=9)
    init = impute_init(r)
    kw = dict(kernel=2) if case == "tma" else dict(exchange="external")
    eng = FilterEngine(d, r, **kw)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd, Md = torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda()
    n = 4 if case == "tma" else 1
    with pytest.raises(_capi.PsmfError):
        eng.run(Yd[:n], Md[:n], Yorig=Yd[:n], E=Md[:n])
    eng.close()


# ---- 4. a forced grid larger than the device holds at once -----------------------------------------------------------
@pytest.mark.parametrize("fused", [False, True], ids=["plain", "eval"])
@pytest.mark.parametrize("r", [1, 16])
def test_forced_grid_above_co_resident_capacity(r, fused):
    """ctas = 4000 on 4000 tiles: the cooperative grid is cut to what fits on the device, and every CTA then holds
    several tiles.  The residual buffer (and the evaluation buffers behind it) must be sized for the grid that runs."""
    d, T, ctas = 128000, 6, 4000
    sms = _sms()
    Y, M, C0, x0, init, E, Yorig, refs = _eval_problem(d, r, None, "f64", True, 2.0, 1, False, seed=128 + r, T=T)
    kw = dict(Yorig=Yorig, E=E) if fused else {}
    res = _engine_run(d, r, Y, M, C0, x0, init, True, ctas=ctas, kernel=1, chunks=[0, 2, T], **kw)
    info = res[4]
    ran = info["ctas"]
    assert info["kernel"] == "direct" and ran < ctas and ran % sms == 0 and ran <= 8 * sms, info
    tiles_per = -(-(d // 32) // ran) + 1
    need = 8 * r * 32 * 8 + tiles_per * 32 * 8 + ((tiles_per * 32 * 17 + 16) if fused else 0)
    assert info["smem_bytes"] >= need, (info, need)
    if fused:
        _check_eval(res, E, refs, None, "f64", False)
    else:
        ost, oX, _, _ = refs[0][0]
        assert relerr(res[0], oX) < 1e-9 and relerr(res[3]["C"], ost.C) < 1e-9


# ---- 5. psmf_eval_full ----------------------------------------------------------------------------------------------
# An engine of several series filters each series in one CTA, whose residual buffer must hold all rows of the series:
# psmf_create refuses such an engine at the row counts that reach the grid-stride loops of the tools (it holds some
# 20 000 rows at r = 16).  Those sizes run with one series; the series strides are covered at d <= MAX_D_SERIES.
MAX_D_SERIES = 4001


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", [1, 5, 8, 9, 16])
@pytest.mark.parametrize("d", [1, 31, 33, 4001, 70000])
def test_eval_full(d, r, tag):
    """Sum over E of (C x_t - yorig_t)^2 with the engine's C and a given X; 70 000 rows are more tile groups than the
    grid (256 groups of 8 tiles): the tile loop strides.  Yorig and E sit in larger buffers (NaN / 1 in the padding)."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    dtype = _dtype(tag)[0]
    rng = np.random.RandomState(d + 17 * r)
    for S, n in ((1, 1), (1, 37)) + (((3, 1), (3, 37)) if d <= MAX_D_SERIES else ()):
        eng = FilterEngine(d, r, n_series=S, dtype=dtype)
        eng.set_state(C_=rng.randn(S, d, r))
        Cg = eng.get_state()["C"].double().cpu().numpy().reshape(S, d, r)
        X = rng.randn(S, n, r)
        Yo = _rounded(rng.randn(S, n, d) * 3.0, tag)
        E = (rng.rand(S, n, d) < 0.3).astype(np.uint8)
        E[:, 0, d - 1] = 1
        Yod, _ = _padded(Yo, dtype, eng.device, pad=3, gap=7, fill=float("nan"))
        Ed, _ = _padded(E, torch.uint8, eng.device, pad=5, gap=11, fill=1)
        out = eng.eval_full(torch.as_tensor(X).cuda(), Yod, Ed).cpu().numpy().reshape(S, 2)
        eng.close()
        for s in range(S):
            sel = E[s] == 1
            ref = float(np.sum(((X[s] @ Cg[s].T) - Yo[s])[sel] ** 2))
            assert out[s, 1] == float(sel.sum()), (S, n, s)
            assert abs(out[s, 0] - ref) <= 1e-12 * ref, (S, n, s, out[s], ref)


# ---- 6. psmf_predict ------------------------------------------------------------------------------------------------
ROLLOUTS = ["identity", "cos", "linear_c", "linear"]


def _predict(eng, n_pred, k0, Xin=None, Xout=None, Yp=None, ldp=0, sst=0):
    from rpsmf_b200 import _capi
    eng._ck(eng._L.psmf_predict(eng._h, n_pred, k0, _ptr(Xin), _ptr(Xout), _ptr(Yp), ldp, sst, _stream()))


@pytest.mark.parametrize("dyn", ROLLOUTS)
@pytest.mark.parametrize("r", RANKS)
def test_rollout(r, dyn):
    """x_k = f(x_{k-1}) for k = k0 .. k0 + n_pred - 1 from the engine's x, against the oracle's dynamics; cos with a
    distinct theta per component and series and k0 up to 10^6 (the kernel keeps the (2 pi theta) k + x order)."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    kind = {"identity": po.DYN_IDENTITY, "cos": po.DYN_COS}.get(dyn, po.DYN_LINEAR)
    rng = np.random.RandomState(r)
    A = 0.9 * np.linalg.qr(rng.randn(r, r))[0]
    c = rng.randn(r) if dyn == "linear_c" else None
    for S in (1, 3):
        eng = FilterEngine(64, r, n_series=S, dynamics=kind)
        if kind == po.DYN_LINEAR:
            eng.set_linear_dynamics(A, c)
        x0, theta = rng.randn(S, r), 0.05 + rng.rand(S, r)
        eng.set_state(x=x0, theta=theta)
        cfg = po.OracleConfig(dynamics=kind, lin_A=A, lin_c=c)
        for n_pred in (1, 50):
            for k0 in (1, 10**6 - n_pred + 1):
                Xp = torch.full((S, n_pred, r), float("nan"), dtype=torch.float64, device="cuda")
                _predict(eng, n_pred, k0, Xout=Xp)
                got = Xp.cpu().numpy()
                for s in range(S):
                    x, ref = x0[s], []
                    for k in range(k0, k0 + n_pred):
                        x = po.dynamics(kind, theta[s], x, k, cfg)[0]
                        ref.append(x)
                    assert relerr(got[s], np.array(ref)) < 1e-12, (S, n_pred, k0, s)
        eng.close()


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("d", [1, 31, 33, 4001, 300000])
def test_projection(d, tag):
    """Ypred = Xpred C' with the engine's C, through the C ABI with ldp > d and a series stride larger than n_pred ldp
    (the padding stays NaN); Xpred_in is copied to Xpred_out bit for bit.  300 000 rows are more tile groups than the
    grid (1024 groups of 8 tiles): the tile loop strides (one series, see MAX_D_SERIES)."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    dtype = _dtype(tag)[0]
    S, n_pred = (3 if d <= MAX_D_SERIES else 1), 5
    rng = np.random.RandomState(d)
    for r in (1, 9, 16):
        eng = FilterEngine(d, r, n_series=S, dtype=dtype)
        eng.set_state(C_=rng.randn(S, d, r))
        Cg = eng.get_state()["C"].double().cpu().numpy().reshape(S, d, r)
        Xin = torch.as_tensor(rng.randn(S, n_pred, r)).cuda()
        Xout = torch.full_like(Xin, float("nan"))
        ldp, sst = d + 3, n_pred * (d + 3) + 13
        buf = torch.full((S * sst,), float("nan"), dtype=dtype, device="cuda")
        Yp = buf.as_strided((S, n_pred, d), (sst, ldp, 1))
        _predict(eng, n_pred, 1, Xin=Xin, Xout=Xout, Yp=buf, ldp=ldp, sst=sst)
        got = Yp.double().cpu().numpy()
        assert torch.equal(Xout, Xin)
        keep = torch.ones_like(buf, dtype=torch.bool)
        keep.as_strided(Yp.shape, Yp.stride()).fill_(False)
        assert bool(buf[keep].isnan().all())
        eng.close()
        ref = np.einsum("skr,sdr->skd", Xin.cpu().numpy(), Cg)
        if tag == "f64":
            assert relerr(got, ref) < 1e-12, r
        else:
            r32 = ref.astype(np.float32)
            assert (np.abs(got - r32) <= np.spacing(np.abs(r32)).astype(np.float64)).all(), r


def test_predict_scratch_roll_out_and_refusals():
    """Xpred_out NULL rolls out into the engine's scratch, which psmf_eval_full shares: after an eval_full the buffer is
    reallocated, and the forecast keeps its bits.  External dynamics without Xpred_in and linear dynamics before
    set_linear_dynamics are refused."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r, S, n_pred = 4001, 16, 3, 50
    rng = np.random.RandomState(5)
    eng = FilterEngine(d, r, n_series=S, dynamics=_capi.DYN_COS)
    eng.set_state(C_=rng.randn(S, d, r), x=rng.randn(S, r), theta=0.05 + rng.rand(S, r))
    Xp = torch.empty((S, n_pred, r), dtype=torch.float64, device="cuda")
    Y1 = torch.empty((S, n_pred, d), dtype=torch.float64, device="cuda")
    _predict(eng, n_pred, 7, Xout=Xp, Yp=Y1, ldp=d, sst=n_pred * d)
    Yo = torch.as_tensor(rng.randn(S, 2, d)).cuda()
    E = torch.ones((S, 2, d), dtype=torch.uint8, device="cuda")
    assert (eng.eval_full(Xp[:, :2], Yo, E)[:, 1] == 2 * d).all()
    Y2 = torch.full_like(Y1, float("nan"))
    _predict(eng, n_pred, 7, Yp=Y2, ldp=d, sst=n_pred * d)
    assert torch.equal(Y1, Y2)
    Y3 = torch.full_like(Y1, float("nan"))
    _predict(eng, n_pred, 7, Xin=Xp, Yp=Y3, ldp=d, sst=n_pred * d)
    assert torch.equal(Y1, Y3)
    eng.close()
    eng = FilterEngine(d, r, dynamics=_capi.DYN_EXTERNAL)
    with pytest.raises(_capi.PsmfError):
        eng.predict(3, 1)
    eng.close()
    eng = FilterEngine(d, r, dynamics=_capi.DYN_LINEAR)
    with pytest.raises(_capi.PsmfError):
        eng.predict(3, 1)
    eng.close()


# ---- 7. handle-free tools, bit for bit -------------------------------------------------------------------------------
SPECIALS = [np.nan, np.inf, -np.inf, -0.0, 0.0, 1e300, -1e300, 3.5e38, 3.40282356e38, 1e-40, 1e-50]


def _special_values(d, n, rng):
    """(d, n) float64: the special values first (NaN, +-inf, -0.0, above FLT_MAX, fp32 subnormal and underflow), then
    random values with about 10 % NaN, shuffled."""
    v = rng.randn(d * n) * 10.0
    v[rng.rand(d * n) < 0.1] = np.nan
    k = min(len(SPECIALS), d * n)
    v[:k] = SPECIALS[:k]
    rng.shuffle(v)
    return v.reshape(d, n)


def _same_bits(got, ref):
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.array_equal(got[ok].view(np.uint8), ref[ok].view(np.uint8))


TOOL_SIZES = [1, 31, 32, 33, 1000]


@pytest.mark.parametrize("n", TOOL_SIZES)
@pytest.mark.parametrize("d", TOOL_SIZES)
def test_ingest_bit_exact(d, n):
    torch = _torch()
    from rpsmf_b200 import _capi
    L = _capi.lib()
    rng = np.random.RandomState(d * 1009 + n)
    src = _special_values(d, n, rng)
    srcd = torch.as_tensor(src).cuda()
    ldy, ldm = d + 3, d + 5
    for tdt, ndt, code in ((torch.float64, np.float64, _capi.F64), (torch.float32, np.float32, _capi.F32)):
        for keep in (0, 1):
            Yb = torch.full((n, ldy), 12345.0, dtype=tdt, device="cuda")
            Mb = torch.full((n, ldm), 7, dtype=torch.uint8, device="cuda")
            _capi.check(None, L.psmf_ingest(0, _ptr(srcd), d, n, code, keep, _ptr(Yb), ldy, _ptr(Mb), ldm, _stream()))
            Yh, Mh = Yb.cpu().numpy(), Mb.cpu().numpy()
            t = src.T
            obs = ~np.isnan(t)
            with np.errstate(over="ignore"):
                ref = np.where(obs | bool(keep), t, 0.0).astype(ndt)
            _same_bits(Yh[:, :d], ref)
            assert np.array_equal(Mh[:, :d], obs.astype(np.uint8))           # inf counts as observed
            assert (Yh[:, d:] == 12345.0).all() and (Mh[:, d:] == 7).all()


@pytest.mark.parametrize("d,n", [(1, 1), (31, 33), (33, 31), (1000, 70), (70, 1000)])
def test_transpose_mask_bit_exact(d, n):
    torch = _torch()
    from rpsmf_b200 import _capi
    rng = np.random.RandomState(d + n)
    src = rng.choice(np.array([0, 1, 2, 255], dtype=np.uint8), size=(d, n))
    ld = d + 4
    dst = torch.full((n, ld), 9, dtype=torch.uint8, device="cuda")
    srcd = torch.as_tensor(src).cuda()
    _capi.check(None, _capi.lib().psmf_transpose_mask(0, _ptr(srcd), d, n, _ptr(dst), ld, _stream()))
    got = dst.cpu().numpy()
    assert np.array_equal(got[:, :d], (src.T != 0).astype(np.uint8))
    assert (got[:, d:] == 9).all()


def _segments_reference(Y, E, starts, seg):
    """common.py:66-75 for one sweep over time-major (n, d) arrays: row i loses the entries j of [s_i, s_i + seg) that
    lie in [0, n) and are not NaN already; returns the number removed."""
    n = Y.shape[0]
    removed = 0
    for i, s in enumerate(starts):
        for j in range(max(int(s), 0), min(int(s) + seg, n)):
            if not np.isnan(Y[j, i]):
                Y[j, i] = np.nan
                E[j, i] = 1
                removed += 1
    return removed


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("d", [1, 255, 257, 1000])
def test_missing_segments_bit_exact(d, tag):
    """Starts below 0, at or beyond n and running past n, a segment longer than n, entries that are NaN or marked in E
    already, and a second sweep over the first; Y and E in larger buffers whose padding stays untouched."""
    torch = _torch()
    from rpsmf_b200 import _capi
    dtype = _dtype(tag)[0]
    ndt = np.float64 if tag == "f64" else np.float32
    n = 60
    rng = np.random.RandomState(d)
    Y = rng.randn(n, d).astype(ndt)
    Y[rng.rand(n, d) < 0.1] = np.nan
    E = (rng.rand(n, d) < 0.05).astype(np.uint8)
    ldy, lde = d + 3, d + 6
    Yb = torch.full((n, ldy), 777.0, dtype=dtype, device="cuda")
    Eb = torch.full((n, lde), 5, dtype=torch.uint8, device="cuda")
    Yb[:, :d] = torch.as_tensor(Y).cuda()
    Eb[:, :d] = torch.as_tensor(E).cuda()
    for seg in (20, n + 15):
        starts = rng.randint(-30, n + 10, size=d).astype(np.int64)
        starts[: min(d, 4)] = [-5, n, n - 3, 0][: min(d, 4)]
        cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
        sd = torch.as_tensor(starts).cuda()
        _capi.check(None, _capi.lib().psmf_missing_segments(0, _capi.F64 if tag == "f64" else _capi.F32, _ptr(Yb), ldy, _ptr(Eb),
                                                            lde, d, n, _ptr(sd), seg, _ptr(cnt), _stream()))
        removed = _segments_reference(Y, E, starts, seg)
        assert int(cnt.item()) == removed, seg
        Yh, Eh = Yb.cpu().numpy(), Eb.cpu().numpy()
        _same_bits(Yh[:, :d], Y)
        assert np.array_equal(Eh[:, :d], E)
        assert (Yh[:, d:] == 777.0).all() and (Eh[:, d:] == 5).all()


@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_count_nan_strided(tag):
    """d n = 700 000 entries, more than the 2048 x 256 threads of the grid; NaN in the padding of the rows is not counted."""
    torch = _torch()
    from rpsmf_b200 import _capi
    dtype = _dtype(tag)[0]
    d, n, ld = 1000, 700, 1005
    rng = np.random.RandomState(11)
    Y = rng.randn(n, d)
    Y[rng.rand(n, d) < 0.07] = np.nan
    Yb = torch.full((n, ld), float("nan"), dtype=dtype, device="cuda")
    Yb[:, :d] = torch.as_tensor(Y).to(dtype).cuda()
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    _capi.check(None, _capi.lib().psmf_count_nan(0, _capi.F64 if tag == "f64" else _capi.F32, _ptr(Yb), ld, d, n, _ptr(cnt),
                                                 _stream()))
    assert int(cnt.item()) == int(np.isnan(Y).sum())
