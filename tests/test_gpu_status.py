"""The first-bad-step report of every kernel (psmf_status / FilterEngine.status) against the float64 oracle.

After a launch the status word holds the smallest step of that launch, counted from 0 and taken over every series of the
engine, at which a series produced a non-finite N / omega / phi / x or N == 0; -1 when there was none.  It is the only way
a caller learns that a run went non-finite: the class surface raises FloatingPointError from it and the imputation
functions blank a sweep's errors with it.

Each case plants a bad value at a known step, steps the float64 oracle on the same data up to its first bad step (which
must be the planted one: a check on the construction, not a hard-coded answer) and asserts that
  * the kernel reports that step, and the variant meant ran (launch_info, as in the kernel matrix);
  * everything written before the bad step -- X, the scalar record, the moment record -- is the clean run's bits, and the
    one-step predictions Yrec up to and including it (Yrec_t = C x_bar_t does not read y_t);
  * every series of the engine that was not poisoned is the clean run's bits in everything;
  * the same engine, its state restored by set_state, then runs the clean data with no report: each launch starts afresh.
Nothing is planted on a step with every row missing in robust mode: the oracle's phi is NaN there by design, while the
kernels define it finite (DESIGN.md).  Batched engines whose series run in waves -- more CTAs or clusters than the device
holds at once -- must still report the earliest bad step, not the one that happened to be written first.
"""

import numpy as np
import pytest

from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import _torch
from test_gpu_kernel_matrix import T, VARIANTS, _check_variant, _dtype, _init, _masked_problem, _rounded, _sms

pytestmark = pytest.mark.gpu

RANKS = [1, 8, 9, 16]
T_BAD = 6
VALUES = {"inf": np.inf, "nan": np.nan, "neginf_nan_mask": -np.inf, "huge": 1e300}
STATE_KEYS = ("C", "P", "V", "Q", "x", "rho", "lam")

# variant -> (kernel-matrix shape it runs on, what it adds to it)
EXTRA = {
    "cluster3": ("direct_S3", "cluster"),            # a thread-block cluster of 3 CTAs per series
    "loglik_direct": ("direct", "loglik"),           # the F_LOGLIK template variant, with the moment record
    "loglik_tma": ("tma_resident", "loglik"),
    "loglik_batch": ("batch8", "loglik"),
    "gradlin_direct": ("direct", "gradlin"),         # F_GRAD_LINEAR under linear dynamics
    "gradlin_tma": ("tma_resident", "gradlin"),
    "gradlin_batch": ("batch8", "gradlin"),
    "eval_direct": ("direct", "eval"),               # fused evaluation
    "eval_batch": ("batch8", "eval"),
    "external_direct": ("direct", "external"),       # external dynamics: one step per launch
    "split_direct": ("direct", "split"),             # caller-driven exchange (run_split), world 1: one step per launch pair
}
ALL = list(VARIANTS) + list(EXTRA)


def _spec(name, r, tag):
    """(kernel-matrix variant, extra, d, S, engine keywords) of a variant."""
    base, extra = EXTRA.get(name, (name, None))
    kernel, d, S, kw = VARIANTS[base]
    if callable(d):
        d = d(r, _dtype(tag)[1])
    kw = dict(kw, kernel=kernel)
    if extra == "cluster":
        kw["ctas"] = 3
    elif extra == "loglik":
        kw["loglik"] = True
    elif extra == "gradlin":
        kw.update(dynamics=2, grad_linear=True)
    elif extra == "external":
        kw["dynamics"] = 3
    elif extra == "split":
        kw.update(exchange="external", ctas=3)
    return base, extra, d, S, kw


def _oracle_first_bad(Y, M, C0, x0, init, cfg, ext=None):
    """First step (0-based) at which the float64 oracle has a non-finite N / omega / phi / x or N == 0, or -1.  Stops there."""
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"], init["lam"])
    with np.errstate(all="ignore"):
        for t in range(Y.shape[0]):
            try:
                st, out = po.step(st, cfg, Y[t], None if M is None else M[t].astype(np.float64), k=1 + t,
                                  xbar_F=None if ext is None else (ext[0][t], ext[1][t]))
            except np.linalg.LinAlgError:
                return t
            if not (np.isfinite([out["N"], out["omega"], out["phi"]]).all() and np.isfinite(st.x).all()) or out["N"] == 0.0:
                return t
    return -1


def _engine(d, r, S, init, C0, x0, tag, kw, lin):
    from rpsmf_b200 import FilterEngine
    eng = FilterEngine(d, r, dtype=_dtype(tag)[0], n_series=S or 1, **kw)
    _restore(eng, init, C0, x0)
    if lin is not None:
        eng.set_linear_dynamics(*lin)
    return eng


def _restore(eng, init, C0, x0):
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=np.atleast_1d(init["rho"]), lam=[init["lam"]])


def _launches(eng, Y, M, chunks, extra, ext=None, ev=None, moments=False):
    """Filter Y (S, T, d) in the launches of `chunks` (one step per launch for external dynamics and run_split).  Returns
    host arrays with the series axis first, the status after every launch, the launch bounds and launch_info."""
    torch = _torch()
    dev, dt = eng.device, eng.dtype
    Sn, Tn, d = Y.shape
    def dev_copy(a, dtype):                  # contiguous on the device: Yorig must have the strides of Y
        return torch.empty(a.shape, dtype=dtype, device=dev).copy_(torch.as_tensor(a))

    Yd = dev_copy(Y, dt)
    Md = None if M is None else dev_copy(M, torch.uint8)
    Ed, Yod = (None, None) if ev is None else (dev_copy(ev[0], torch.uint8), dev_copy(ev[1], dt))
    if extra in ("external", "split"):
        chunks = list(range(Tn + 1))
    acc = dict(X=[], Yrec=[], scal=[], mom=[])
    status, evsum = [], None
    for a, b in zip(chunks[:-1], chunks[1:]):
        rk = dict(want_X=True, want_Yrec=True, want_scal=True, want_moments=moments, want_grad=extra == "gradlin")
        if ext is not None:
            rk.update(xbar=ext[0][:, a], F=ext[1][:, a])
        if ev is not None:
            rk.update(E=Ed[:, a:b], Yorig=Yod[:, a:b])
        Ya, Ma = Yd[:, a:b], None if Md is None else Md[:, a:b]
        out = eng.run_split(Ya, Ma, 1 + a, lambda buf: None, **rk) if extra == "split" else eng.run(Ya, Ma, k0=1 + a, **rk)
        status.append(eng.status())
        n = b - a
        acc["X"].append(out["X"].reshape(Sn, n, -1).cpu().numpy())
        acc["Yrec"].append(out["Yrec"].reshape(Sn, n, d).double().cpu().numpy())
        acc["scal"].append(out["scal"].reshape(Sn, n, -1).cpu().numpy())
        if moments:
            acc["mom"].append(out["moments"].reshape(Sn, n, -1).cpu().numpy())
        if ev is not None:
            e = out["eval"].reshape(Sn, -1).cpu().numpy()
            evsum = e if evsum is None else evsum + e
    res = {k: np.concatenate(v, axis=1) for k, v in acc.items() if v}
    st = eng.get_state()
    for k in STATE_KEYS:
        res[k] = st[k].double().cpu().numpy().reshape(Sn, -1)
    res.update(eval=evsum, status=status, chunks=chunks, info=eng.launch_info())
    return res


def _expected(chunks, t):
    """Status after each launch up to the one that holds step t: -1, then t relative to that launch."""
    out = []
    for a, b in zip(chunks[:-1], chunks[1:]):
        if t < b:
            return out + [t - a]
        out.append(-1)
    return out


def _bits_before(clean, bad, s, t):
    for k in ("X", "scal", "mom"):
        if k in clean:
            assert np.array_equal(bad[k][s, :t], clean[k][s, :t]), (k, s, t)
    assert np.array_equal(bad["Yrec"][s, :t + 1], clean["Yrec"][s, :t + 1]), ("Yrec", s, t)


def _bits_all(clean, bad, sel):
    for k in ("X", "Yrec", "scal", "mom", "eval") + STATE_KEYS:
        if k in clean and clean[k] is not None:
            assert np.array_equal(bad[k][sel], clean[k][sel]), k


def _problem(base, extra, d, S, r, tag, seed=None):
    """Inputs of a variant with the series axis first: (Y, M, C0, x0, init, oracle config keywords, lin, ext, ev)."""
    Y, M, C0, x0, _ = _masked_problem(d, r, S, seed=100 * r + d % 97 if seed is None else seed)
    init = _init(r, d, VARIANTS[base][3].get("rho_vector", False))
    if S is None:
        Y, M, C0, x0 = Y[None], M[None], C0[None], x0[None]
    Y, C0 = _rounded(Y, tag), _rounded(C0, tag)
    Sn = Y.shape[0]
    rng = np.random.RandomState(r)
    cfg, lin, ext, ev = dict(robust=True), None, None, None
    if extra == "gradlin":
        lin = (0.9 * np.eye(r) + 0.02 * rng.randn(r, r), 0.05 * rng.randn(r))
        cfg.update(dynamics=po.DYN_LINEAR, lin_A=lin[0], lin_c=lin[1])
    elif extra == "external":
        ext = (rng.rand(Sn, T, r), 0.9 * np.eye(r) + 0.01 * rng.randn(Sn, T, r, r))
    elif extra == "eval":
        ev = (((rng.rand(Sn, T, d) < 0.15) & (M == 0)).astype(np.uint8), Y + 0.1 * rng.randn(Sn, T, d))
    return Y, M, C0, x0, init, cfg, lin, ext, ev


def _poisoned_vs_clean(spec, r, tag, trigger, plants, chunks=(0, T), prob=None):
    """Plant VALUES[trigger] at (series, step) for each of `plants` in one observed entry, run the poisoned and then, on the
    same engine with its state restored, the clean data; check the report against the oracle and the bits against the clean
    run.  Returns the poisoned run."""
    base, extra, d, S, kw = spec
    esize = _dtype(tag)[1]
    nan_mask = trigger == "neginf_nan_mask"
    Y, M, C0, x0, init, cfg, lin, ext, ev = prob if prob is not None else _problem(base, extra, d, S, r, tag)
    if nan_mask:
        kw = dict(kw, nan_mask=True)
        Yc, Mc = np.where(M != 0, Y, np.nan), None
    else:
        Yc, Mc = Y, M
    Yb, Mb = Yc.copy(), None if Mc is None else Mc.copy()
    row = d // 3
    for s, t in plants:
        Yb[s, t, row] = VALUES[trigger]
        if Mb is not None:
            Mb[s, t, row] = 1
    # the reference: the oracle on the poisoned series fails first at the planted step
    for s, t in plants:
        Yo, Mo = (np.where(np.isnan(Yb[s]), 0.0, Yb[s]), ~np.isnan(Yb[s])) if nan_mask else (Yb[s], Mb[s])
        got = _oracle_first_bad(Yo, Mo, C0[s], x0[s], init, po.OracleConfig(**cfg), None if ext is None else (ext[0][s], ext[1][s]))
        assert got == t, (s, t, got)
    tmin = min(t for _, t in plants)
    moments = extra == "loglik"
    eng = _engine(d, r, S, init, C0 if S else C0[0], x0 if S else x0[0], tag, kw, lin)
    try:
        bad = _launches(eng, Yb, Mb, list(chunks), extra, ext, ev, moments)
        _restore(eng, init, C0 if S else C0[0], x0 if S else x0[0])
        clean = _launches(eng, Yc, Mc, list(chunks), extra, ext, ev, moments)
    finally:
        eng.close()
    for res in (bad, clean):
        _check_variant(base, res["info"], r, esize, d)
        if extra == "cluster":
            assert res["info"]["ctas"] == 3, res["info"]
    if moments:
        assert clean["scal"].shape[-1] == 10
    exp = _expected(bad["chunks"], tmin)
    assert bad["status"][:len(exp)] == exp, (bad["status"], exp)
    assert clean["status"] == [-1] * len(clean["status"]), clean["status"]
    poisoned = sorted({s for s, _ in plants})
    for s in poisoned:
        _bits_before(clean, bad, s, min(t for q, t in plants if q == s))
    others = np.setdiff1d(np.arange(Y.shape[0]), poisoned)
    if others.size:
        _bits_all(clean, bad, others)
    return bad


def _series_mid(S):
    return 0 if S is None else S // 2


# ---- a. every kernel, every trigger -------------------------------------------------------------------------------------
A_PARAMS = [(n, r, tag, trig) for n in ALL for r in RANKS for tag in ("f64", "f32")
            for trig in ("inf", "nan", "neginf_nan_mask") + (("huge",) if tag == "f64" else ())]


@pytest.mark.parametrize("name,r,tag,trigger", A_PARAMS, ids=["%s-r%d-%s-%s" % p for p in A_PARAMS])
def test_bad_step_on_every_kernel(name, r, tag, trigger):
    """+inf, NaN (byte mask), -inf (NaN-encoded mask) at one observed entry, or, robust f64, 1e300: finite data whose
    square overflows, so omega is inf."""
    spec = _spec(name, r, tag)
    _poisoned_vs_clean(spec, r, tag, trigger, [(_series_mid(spec[3]), T_BAD)])


# ---- b. what is not bad ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("name", ALL)
def test_missing_data_is_not_bad(name, tag):
    """NaN-encoded missing entries (a whole NaN row, a whole NaN step among them) and a step with every row missing under the
    byte mask (V != 0: a pure prediction step) report nothing."""
    r = 9
    base, extra, d, S, kw = _spec(name, r, tag)
    Y, M, C0, x0, init, cfg, lin, ext, ev = _problem(base, extra, d, S, r, tag)
    Mz = M.copy()
    Mz[:, 4] = 0
    Mz[:, :, 5] = 0
    Yn = np.where(Mz != 0, Y, np.nan)
    for Yi, Mi, nan_mask in ((Yn, None, True), (Y * Mz, Mz, False)):
        eng = _engine(d, r, S, init, C0 if S else C0[0], x0 if S else x0[0], tag, dict(kw, nan_mask=nan_mask), lin)
        try:
            res = _launches(eng, Yi, Mi, [0, 5, T], extra, ext, ev, extra == "loglik")
        finally:
            eng.close()
        _check_variant(base, res["info"], r, _dtype(tag)[1], d)
        assert res["status"] == [-1] * len(res["status"]), (nan_mask, res["status"])
        assert np.isfinite(res["X"]).all() and np.isfinite(res["C"]).all()


# ---- c. N == 0 ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("name", ALL)
def test_zero_N_is_bad(name, tag):
    """PSMF with V = 0 and one step t > 0 with every row missing: a = x_bar' V x_bar = 0 and eta = 0, so N = a + eta = 0."""
    r, t = 9, 5
    base, extra, d, S, kw = _spec(name, r, tag)
    Y, M, C0, x0, init, cfg, lin, ext, ev = _problem(base, extra, d, S, r, tag)
    init = dict(init, V=np.zeros((r, r)), lam=0.0)
    cfg = dict(cfg, robust=False)
    M = np.ones_like(M)                      # the zeros of Y are observed zeros now
    M[:, t] = 0
    Y = Y.copy()
    Y[:, t] = 0.0
    for s in range(Y.shape[0]):
        got = _oracle_first_bad(Y[s], M[s], C0[s], x0[s], init, po.OracleConfig(**cfg), None if ext is None else (ext[0][s], ext[1][s]))
        assert got == t, (s, got)
    eng = _engine(d, r, S, init, C0 if S else C0[0], x0 if S else x0[0], tag, dict(kw, robust=False), lin)
    try:
        res = _launches(eng, Y, M, [0, T], extra, ext, ev, extra == "loglik")
    finally:
        eng.close()
    _check_variant(base, res["info"], r, _dtype(tag)[1], d)
    exp = _expected(res["chunks"], t)
    assert res["status"][:len(exp)] == exp, (res["status"], exp)


# ---- d. launch splits --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", RANKS)
@pytest.mark.parametrize("name", ["direct", "tma_resident", "batch8"])
def test_bad_step_is_launch_relative(name, r, tag):
    """A bad value at absolute step 7 filtered in the launches [0, 5) and [5, 12): the first reports nothing, the second 2."""
    spec = _spec(name, r, tag)
    bad = _poisoned_vs_clean(spec, r, tag, "inf", [(_series_mid(spec[3]), 7)], chunks=(0, 5, T))
    assert bad["status"] == [-1, 2]


# ---- e. several bad series: the earliest step wins ----------------------------------------------------------------------------
MULTI = [n for n in ALL if VARIANTS[EXTRA.get(n, (n,))[0]][2] is not None]


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", [1, 9, 16])
@pytest.mark.parametrize("name", MULTI)
def test_earliest_of_several_bad_series(name, r, tag):
    """Series 0 goes bad at step 9 and series 2 at step 3; series 1 is untouched and keeps the clean run's bits."""
    spec = _spec(name, r, tag)
    bad = _poisoned_vs_clean(spec, r, tag, "inf", [(0, 9), (2, 3)])
    assert bad["status"][0] == 3


def _wave_plants(S):
    """Series 0 at step T - 2 (first wave), the last 8 series at step 1 (last wave), a few in between at steps in between."""
    return [(0, T - 2), (S // 4, 8), (S // 2, 5), (3 * S // 4, 3)] + [(s, 1) for s in range(S - 8, S)]


def _resident_bound(info):
    """An upper bound of the CTAs the device holds at once: threads, dynamic shared memory (227 KB a block on a B200) and 32
    blocks per SM."""
    return _sms() * min(2048 // info["threads"], 232448 // max(1, info["smem_bytes"]), 32)


def _wave_case(base, d, S, kw, r=8, tag="f64"):
    spec = (base, None, d, S, dict(kw))
    Y, M, C0, x0 = make_problem(d, r, T, seed=d + S, S=S)
    prob = (_rounded(Y, tag), M, _rounded(C0, tag), x0, impute_init(r), dict(robust=True), None, None, None)
    bad = _poisoned_vs_clean(spec, r, tag, "inf", _wave_plants(S), prob=prob)
    assert bad["status"] == [1]
    return bad["info"]


def test_batch_kernel_in_waves_reports_the_earliest_step():
    S = 32 * _sms()
    info = _wave_case("batch4", 203, S, dict(kernel=3))
    assert info["threads"] == 128 and S > _resident_bound(info), info


def test_clusters_in_waves_report_the_earliest_step():
    torch = _torch()
    S, c = 40, 16
    info = _wave_case("direct_S3", 6000, S, dict(kernel=1, ctas=c))
    assert info["kernel"] == "direct" and info["ctas"] == c, info
    assert S * c > torch.cuda.get_device_properties(0).multi_processor_count * 2


def test_direct_kernel_in_waves_reports_the_earliest_step():
    S = 8 * _sms() + 16
    info = _wave_case("direct_S3", 1100, S, dict(kernel=1))
    assert info["kernel"] == "direct" and info["ctas"] == 1 and S > _resident_bound(info), info


# ---- f. host surfaces ------------------------------------------------------------------------------------------------------------
def _finite_only(theta, x, t):
    """A plain callable (the external-dynamics path) that refuses a non-finite state, as a user's model may."""
    x = np.asarray(x)
    if not np.all(np.isfinite(x)):
        raise ValueError("nonlinearity called on a non-finite state")
    return 0.9 * np.tanh(x) + 0.01 * np.asarray(theta).reshape(x.shape)


def _nonlinearity(kind, r):
    from rpsmf_b200.nonlinearities import RandomWalk, affine, cos_phase
    if kind == "random_walk":
        return RandomWalk(), np.zeros((1, 1))
    theta = 0.05 + 0.1 * np.random.RandomState(r).rand(r, 1)
    if kind == "cos":
        return cos_phase, theta
    if kind == "affine":
        return affine(lambda th, x, t: 0.9 * np.asarray(x) + 0.01 * np.asarray(th).reshape(np.shape(x))), theta
    return _finite_only, theta


def _ydict(Y):
    return {k + 1: Y[k].reshape(-1, 1) for k in range(Y.shape[0])}


def _class_problem(k_bad, d=40, r=3, n=20):
    Y, _, C0, x0 = make_problem(d, r, n, seed=11, missing=0.0)
    Y[k_bad - 1, 5] = np.inf                 # absolute step k_bad, 1-based as pypsmf counts
    return Y, C0, x0


@pytest.mark.parametrize("kind", ["random_walk", "cos", "affine", "callable"])
@pytest.mark.parametrize("robust", [False, True], ids=["PSMFIter", "rPSMFIter"])
def test_class_surface_names_the_bad_step(robust, kind):
    from rpsmf_b200 import PSMFIter, _capi, rPSMFIter
    k, r = 9, 3
    Y, C0, x0 = _class_problem(k, r=r)
    n, d = Y.shape
    nl, theta0 = _nonlinearity(kind, r)
    init = impute_init(r)
    if robust:
        o = rPSMFIter(theta0, C0, init["V"], x0.reshape(r, 1), init["P"], init["Q"], init["rho"] * np.eye(d), init["lam"], nl)
    else:
        o = PSMFIter(theta0, C0, init["V"], x0.reshape(r, 1), init["P"], {i: init["Q"] for i in range(n + 1)},
                     {i: init["rho"] * np.eye(d) for i in range(n + 1)}, nl)
    want = {"random_walk": _capi.DYN_IDENTITY, "cos": _capi.DYN_COS, "affine": _capi.DYN_LINEAR, "callable": _capi.DYN_EXTERNAL}
    assert o._dyn == want[kind]
    try:
        with pytest.raises(FloatingPointError, match=r"at step %d$" % k):
            o.step(_ydict(Y), 1, n)
    finally:
        o.close()


def test_recursive_class_names_the_bad_step_of_a_later_block():
    """update_every = 7: step 10 lies in the second block, [8, 14]."""
    from rpsmf_b200 import rPSMFRecursive
    from rpsmf_b200.nonlinearities import cos_phase
    k, r = 10, 3
    Y, C0, x0 = _class_problem(k, r=r)
    n, d = Y.shape
    init = impute_init(r)
    o = rPSMFRecursive(0.05 * np.ones((r, 1)), C0, init["V"], x0.reshape(r, 1), init["P"], init["Q"], init["rho"] * np.eye(d),
                       init["lam"], cos_phase)
    try:
        with pytest.raises(FloatingPointError, match=r"at step %d$" % k):
            o.run(_ydict(Y), n, 0, update_every=7)
    finally:
        o.close()


def test_statespace_names_the_zero_based_column():
    from rpsmf_b200 import statespace
    r, m, n, col = 2, 30, 15, 6
    s = 2 * r
    rng = np.random.RandomState(3)
    Y = rng.randn(m, n)
    Y[4, col] = np.inf
    A = 0.9 * np.eye(s)
    H = np.hstack([np.eye(r), np.zeros((r, r))])
    X = np.zeros((s, n))
    with pytest.raises(FloatingPointError, match=r"at step %d$" % col):
        statespace.PSMF(r, Y, 0.1 * np.eye(s), A, 0.5 * np.eye(m), H, np.eye(r), np.eye(s), rng.rand(m, r), X, m, n)


def _impute_inputs(seed, d=50, n=30, r=3):
    rng = np.random.RandomState(seed)
    Yorig = rng.randn(r, n).cumsum(axis=1)
    Yorig = rng.rand(d, r) @ Yorig + 0.1 * rng.randn(d, n)
    Mmiss = (rng.rand(d, n) < 0.1).astype(np.float64)
    M = 1.0 - Mmiss
    return Yorig * M, M, Mmiss, Yorig, rng.rand(d, r), rng.rand(r, n)


def test_robust_psmf_blanks_the_poisoned_sweep():
    from rpsmf_b200.impute import robust_PSMF
    d, n, r = 50, 30, 3
    Y, M, Mmiss, Yorig, C, X = _impute_inputs(1, d, n, r)
    init = impute_init(r)
    args = (init["V"], init["Q"], init["rho"], init["P"], init["lam"], 2.0, 2, Yorig, 1.0)
    Ep, Ef, _, _ = robust_PSMF(Y, C, X.copy(), d, n, r, M, Mmiss, *args)
    assert np.isfinite(Ep).all() and np.isfinite(Ef).all()
    Yb = Y.copy()
    row = int(np.argmax(M[:, 12]))           # an observed entry
    Yb[row, 12] = np.inf
    Ep, Ef, _, _ = robust_PSMF(Yb, C, X.copy(), d, n, r, M, Mmiss, *args)
    assert Ep[0, 0] == 1.0 and Ef[0, 0] == 1.0
    assert np.isnan(Ep[0, 1:]).all() and np.isnan(Ef[0, 1:]).all()


def test_fit_repeats_blanks_only_the_poisoned_repeat():
    from rpsmf_b200.impute import fit_repeats
    d, n, r, S, bad = 50, 30, 3, 4, 2
    ins = [_impute_inputs(10 + k, d, n, r) for k in range(S)]
    Yorig = ins[0][3]
    Ys, Ms, Mmisses = [], [], []
    for k in range(S):
        # the same data set for every repeat (each its own mask and initial C, X), as in the experiment
        Mmiss = ins[k][2]
        Ys.append(Yorig * (1.0 - Mmiss)); Ms.append(1.0 - Mmiss); Mmisses.append(Mmiss)
    init = impute_init(r)

    def fit(Ys):
        return fit_repeats(Ys, [i[4] for i in ins], [i[5].copy() for i in ins], Ms, Mmisses, init["V"], init["Q"], init["rho"],
                           init["P"], init["lam"], 2.0, 2, Yorig, [1.0] * S)

    Ep0, Ef0, _, In0 = fit(Ys)
    Yb = [y.copy() for y in Ys]
    row = int(np.argmax(Ms[bad][:, 12]))
    Yb[bad][row, 12] = np.inf
    Ep, Ef, _, In = fit(Yb)
    assert np.isnan(Ep[bad][0, 1:]).all() and np.isnan(Ef[bad][0, 1:]).all()
    for k in range(S):
        assert np.isfinite(Ep0[k]).all() and np.isfinite(Ef0[k]).all()
        if k != bad:
            assert np.array_equal(Ep[k], Ep0[k]) and np.array_equal(Ef[k], Ef0[k]) and In[k] == In0[k], k
