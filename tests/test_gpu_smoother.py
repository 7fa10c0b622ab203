# -*- coding: utf-8 -*-
"""Per-step moment record (psmf_set_moments) of every filter kernel and the fixed-interval smoother (psmf_smooth).

Each case forces its kernel and checks from launch_info() that the variant it meant to test ran.  The record is compared with
the float64 restatement of tests/smoother_oracle.py on the oracle's trajectory (fp64 1e-9, fp32 storage 1e-4 on fp32-rounded
Y and C0); psmf_smooth is compared with the restatement applied to the GPU's own record (1e-12), which isolates the backward
kernel, and the smoothed states with the restatement on the oracle's record.  The restatement itself is checked against the
dense joint posterior in tests/test_smoother_cpu.py."""

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
import smoother_oracle as so
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _padded, _torch
from test_gpu_kernel_matrix import KERNEL_KW, KNAME, SPLIT_RANKS, TOL32, VARIANTS as KM_VARIANTS, _check_variant

pytestmark = pytest.mark.gpu

T = 12
CHUNKS = [0, 5, 12]                # two launches, each writing through a view advanced by the steps before it
RANKS = [1, 5, 8, 9, 16]
VARIANTS = {k: KM_VARIANTS[k] for k in ("direct", "direct_S3", "rhovec", "rhovec_S3", "tma_resident", "tma_stream", "batch8", "batch4")}
VARIANTS["rhovec_S1"] = KM_VARIANTS["rhovec"]
VARIANTS["cluster"] = (1, 4001, 3, dict(ctas=3))          # a thread-block cluster of 3 CTAs per series
VARIANTS.pop("rhovec")


def _init(r, d, rho_vector, seed=0):
    init = impute_init(r)
    if rho_vector:
        init["rho"] = 10.0 * (0.5 + np.random.RandomState(seed).rand(d))
    return init


def _masked(d, r, S, seed, T_=T):
    Y, M, C0, x0 = make_problem(d, r, T_, seed=seed, S=S)
    M[..., [1, d // 2]] = 0
    M[..., T_ - 1, :] = 0       # a step with every row missing, the last (the robust oracle's V is NaN after it, 0 * inf)
    return Y * M, M, C0, x0


def _engine(d, r, init, C0, x0, S=None, A=None, c=None, theta=None, **kw):
    from rpsmf_b200 import FilterEngine
    eng = FilterEngine(d, r, n_series=S or 1, **kw)
    rho = init["rho"]
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=rho if np.ndim(rho) else [rho], lam=[init["lam"]],
                  theta=theta)
    if A is not None:
        eng.set_linear_dynamics(A, c)
    return eng


def _run(d, r, Y, M, C0, x0, init, S=None, chunks=CHUNKS, dtype=None, moments=True, nan=False, want_grad=False, want_scal=True,
         E=None, Yorig=None, A=None, c=None, theta=None, keep=False, **kw):
    """Filter Y in the launches of `chunks`, the moment record of all of them in one (S, T, NMOM) horizon."""
    torch = _torch()
    dtype = dtype or torch.float64
    eng = _engine(d, r, init, C0, x0, S=S, A=A, c=c, theta=theta, dtype=dtype, nan_mask=nan, **kw)
    one = S is None
    Yh = Y[None] if one else Y
    if nan:
        Yh = np.where((M[None] if one else M) == 0, np.nan, Yh)
    Yd = _padded(Yh, dtype, eng.device)[0]
    Md = None if (M is None or nan) else _padded(M[None] if one else M, torch.uint8, eng.device)[0]
    Ed = None if E is None else _padded(E[None] if one else E, torch.uint8, eng.device)[0]
    Yod = None if Yorig is None else _padded(Yorig[None] if one else Yorig, dtype, eng.device)[0]
    Tn = Yd.shape[1]
    mom = torch.full((S or 1, Tn, so.nmom(r)), float("nan"), dtype=torch.float64, device=eng.device) if moments else None
    res = dict(X=[], scal=[], Yrec=[], grad=[], eval=[], status=[])
    for a, b in zip(chunks[:-1], chunks[1:]):
        ev = {} if Ed is None else dict(E=Ed[:, a:b], Yorig=Yod[:, a:b])
        out = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, want_Yrec=True, want_scal=want_scal,
                      want_grad=want_grad, moments_out=None if mom is None else mom[:, a:b], **ev)
        res["status"].append(eng.status())
        for k in ("X", "scal", "Yrec", "eval"):
            if k in out:
                res[k].append(out[k].double().cpu().numpy().reshape((S or 1, b - a, -1) if k != "eval" else (S or 1, -1)))
        if want_grad:
            g = [out["grad_A"].reshape(S or 1, -1), out["grad_c"].reshape(S or 1, -1)] if "grad_A" in out else [out["grad"].reshape(S or 1, -1)]
            res["grad"].append(torch.cat(g, dim=1).cpu().numpy())
    for k in ("X", "scal", "Yrec"):
        res[k] = np.concatenate(res[k], axis=1) if res[k] else None
    res["state"] = {k: (v.double().cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()}
    res["info"] = eng.launch_info()
    res["mom"] = mom
    if keep:
        res["engine"] = eng
    else:
        res["engine"] = None
        if mom is not None:
            Xs, Ps = eng.smooth(mom, want_P=True)
            res["Xs"] = Xs.reshape(S or 1, Tn, r).cpu().numpy()
            res["Ps"] = Ps.reshape(S or 1, Tn, r, r).cpu().numpy()
            res["Xs_noP"] = eng.smooth(mom).reshape(S or 1, Tn, r).cpu().numpy()
        res["mom"] = None if mom is None else mom.cpu().numpy()
        eng.close()
    return res


def _rounded(a, f32):
    return a.astype(np.float32).astype(np.float64) if f32 else a


def _oracle_record(Y, M, C0, x0, init, f32=False, theta=None, **cfgkw):
    cfg = po.OracleConfig(c_update_transpose=cfgkw.pop("c_update_transpose", True), **cfgkw)
    rho = init["rho"]
    st = po.OracleState(_rounded(C0, f32).copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(),
                        rho if np.ndim(rho) == 0 else np.array(rho), init["lam"], None if theta is None else np.asarray(theta, float))
    return so.record_run(st, cfg, _rounded(Y, f32), M)[1]


def _check(res, Y, M, C0, x0, init, tol, S=None, f32=False, **cfgkw):
    r = C0.shape[-1]
    for s in range(S or 1):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        ref = _oracle_record(one(Y), one(M), one(C0), one(x0), init, f32=f32, **cfgkw)
        mom = res["mom"][s]
        assert relerr(mom, ref) < tol, (s, relerr(mom, ref))
        # the backward kernel against the restatement on the GPU's own record, with and without Ps_out
        Xg, Pg = so.rts(mom, r)
        assert relerr(res["Xs"][s], Xg) < 1e-12 and relerr(res["Ps"][s], Pg) < 1e-12
        assert np.array_equal(res["Xs_noP"][s], res["Xs"][s])
        Xo, Po = so.rts(ref, r)
        assert relerr(res["Xs"][s], Xo) < tol and relerr(res["Ps"][s], Po) < tol
        # the record's x_t is the filtered X of the run
        assert np.array_equal(mom[:, so.nmom(r) - r * r - r:so.nmom(r) - r * r], res["X"][s])


MATRIX = [(v, r, tag) for v in VARIANTS for r in RANKS for tag in ("f64", "f32")]


@pytest.mark.parametrize("name,r,tag", MATRIX, ids=["%s-r%d-%s" % p for p in MATRIX])
def test_record_and_smoother_against_oracle(name, r, tag):
    torch = _torch()
    kernel, d, S, kw = VARIANTS[name]
    f32 = tag == "f32"
    esize = 4 if f32 else 8
    if callable(d):
        d = d(r, esize)
    Y, M, C0, x0 = _masked(d, r, S, seed=1200 + 7 * r + d % 89)
    init = _init(r, d, kw.get("rho_vector", False))
    res = _run(d, r, Y, M, C0, x0, init, S=S, kernel=kernel, dtype=torch.float32 if f32 else torch.float64, **kw)
    if name == "cluster":
        assert res["info"]["kernel"] == "direct" and res["info"]["ctas"] == 3, res["info"]
    else:
        _check_variant(name.replace("_S1", ""), res["info"], r, esize, d)
    assert res["status"] == [-1, -1]
    _check(res, Y, M, C0, x0, init, TOL32 if f32 else TOL, S=S, f32=f32, robust=True)


@pytest.mark.parametrize("S", [None, 3], ids=["S1", "S3"])
@pytest.mark.parametrize("r", [1, 8, 16], ids=lambda r: "r%d" % r)
def test_smoother_across_chunks(r, S):
    """T = 53: the backward walk crosses three chunk boundaries of psmf_smooth (16 steps each) and ends in a 4-step tail
    chunk; x^s and P^s are carried from chunk to chunk in shared memory and the gain buffer is reused."""
    Tl = 53
    d = 700
    Y, M, C0, x0 = _masked(d, r, S, seed=400 + r, T_=Tl)
    init = _init(r, d, False)
    res = _run(d, r, Y, M, C0, x0, init, S=S, chunks=[0, 20, Tl], kernel=1, robust=True)
    assert res["status"] == [-1, -1] and res["info"]["kernel"] == "direct"
    for s in range(S or 1):
        mom = res["mom"][s]
        assert np.isfinite(mom).all()
        Xg, Pg = so.rts(mom, r)
        assert relerr(res["Xs"][s], Xg) < 1e-12 and relerr(res["Ps"][s], Pg) < 1e-12
        assert np.array_equal(res["Xs_noP"][s], res["Xs"][s])
        # each chunk boundary on its own: the steps next to it (t = 36 / 37, 20 / 21, 4 / 5) are smoothed like the rest
        for t in (4, 5, 20, 21, 36, 37, 51):
            assert relerr(res["Xs"][s][t], Xg[t]) < 1e-11, t
    ref = _oracle_record(Y if S is None else Y[0], M if S is None else M[0], C0 if S is None else C0[0], x0 if S is None else x0[0],
                         init, robust=True)
    Xo, Po = so.rts(ref, r)
    assert relerr(res["Xs"][0], Xo) < TOL and relerr(res["Ps"][0], Po) < TOL


@pytest.mark.parametrize("dyn", ["identity", "linear"])
@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
def test_smoother_equals_dense_posterior(dyn, kernel):
    """PSMF with V = 0 is a linear-Gaussian model: the smoothed X is the dense joint posterior of x_{1:T}."""
    torch = _torch()
    r, d = 5, 960
    Y, M, C0, x0 = make_problem(d, r, T, seed=77)
    M[:, [3, 400]] = 0
    M[6, ::2] = 0              # (a step with every row missing has N = a + eta = 0 when V = 0: the filter flags it)
    Y = Y * M
    rng = np.random.RandomState(5)
    B = rng.randn(r, r)
    init = dict(impute_init(r), V=np.zeros((r, r)), Q=0.05 * (B @ B.T / r + np.eye(r)), P=np.eye(r), rho=0.5, lam=0.0)
    A, c = (0.9 * np.linalg.qr(rng.randn(r, r))[0], 0.1 * rng.randn(r)) if dyn == "linear" else (None, None)
    from rpsmf_b200 import _capi
    res = _run(d, r, Y, M, C0, x0, init, robust=False, dynamics=_capi.DYN_LINEAR if dyn == "linear" else 0, A=A, c=c,
               **KERNEL_KW[kernel])
    assert res["info"]["kernel"] == KNAME[kernel] and res["status"] == [-1, -1]
    Ad, cd = (A, c) if dyn == "linear" else (np.eye(r), np.zeros(r))
    Xd, Pd = so.dense_posterior(C0, 0.5, init["Q"], Ad, cd, x0, init["P"], Y, M)
    assert relerr(res["Xs"][0], Xd) < 1e-9
    assert relerr(res["Ps"][0], Pd) < 1e-9


def _dynamics(r, seed):
    rng = np.random.RandomState(seed)
    return 0.9 * np.eye(r) + 0.1 * rng.randn(r, r) / np.sqrt(r), 0.1 * rng.randn(r)


def _theta(r):
    return 0.05 + 0.1 * np.random.RandomState(r).rand(r)


FLAG_CASES = {
    # id: (engine keywords, oracle keywords)
    "psmf_vt": (dict(robust=False, c_update_transpose=True), dict(robust=False, c_update_transpose=True)),
    "psmf_vtt": (dict(robust=False, c_update_transpose=False), dict(robust=False, c_update_transpose=False)),
    "fixed_lambda": (dict(robust=True, fixed_lambda=True), dict(robust=True, fixed_lambda=True)),
    "alpha_beta": (dict(robust=True, alpha=0.97, beta=1.06), dict(robust=True, alpha=0.97, beta=1.06)),
    "cos": (dict(robust=True, dynamics=1), dict(robust=True, dynamics=po.DYN_COS)),
    "linear": (dict(robust=True, dynamics=2), dict(robust=True, dynamics=po.DYN_LINEAR)),
    "loglik": (dict(robust=True, loglik=True), dict(robust=True)),
    "grad_linear": (dict(robust=True, dynamics=2, grad_linear=True), dict(robust=True, dynamics=po.DYN_LINEAR)),
    "grad_linear_loglik": (dict(robust=True, dynamics=2, grad_linear=True, loglik=True), dict(robust=True, dynamics=po.DYN_LINEAR)),
}


@pytest.mark.parametrize("case", list(FLAG_CASES))
@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("r", SPLIT_RANKS, ids=lambda r: "r%d" % r)
def test_flags_and_dynamics(case, kernel, r):
    ekw, okw = FLAG_CASES[case]
    d = 960 if kernel != 3 else 203
    Y, M, C0, x0 = _masked(d, r, None, seed=31 * r + kernel)
    init = _init(r, d, False)
    extra = {}
    if ekw.get("dynamics") == 2:
        A, c = _dynamics(r, r)
        extra = dict(A=A, c=c)
        okw = dict(okw, lin_A=A, lin_c=c)
    theta = _theta(r) if ekw.get("dynamics") == 1 else None
    res = _run(d, r, Y, M, C0, x0, init, theta=theta, want_grad=case.startswith("grad") or case == "cos", **ekw, **extra,
               **KERNEL_KW[kernel])
    assert res["info"]["kernel"] == KNAME[kernel]
    assert res["scal"].shape[-1] == (10 if ekw.get("loglik") else 8)
    _check(res, Y, M, C0, x0, init, TOL, theta=theta, **okw)


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("r", SPLIT_RANKS, ids=lambda r: "r%d" % r)
def test_nan_mask_record_is_bit_identical(kernel, r):
    d = 960 if kernel != 3 else 203
    Y, M, C0, x0 = _masked(d, r, None, seed=5 * r)
    init = _init(r, d, False)
    a = _run(d, r, Y, M, C0, x0, init, **KERNEL_KW[kernel])
    b = _run(d, r, Y, M, C0, x0, init, nan=True, **KERNEL_KW[kernel])
    assert a["info"]["kernel"] == b["info"]["kernel"] == KNAME[kernel]
    assert np.array_equal(a["mom"], b["mom"], equal_nan=True) and np.array_equal(a["Xs"], b["Xs"])


@pytest.mark.parametrize("r", SPLIT_RANKS, ids=lambda r: "r%d" % r)
def test_external_dynamics_record_equals_cos(r):
    """External dynamics, one step per run, fed with the cos dynamics' x_bar and F: the record equals the cos run's."""
    torch = _torch()
    d = 960
    Y, M, C0, x0 = _masked(d, r, None, seed=3 * r)
    init = _init(r, d, False)
    th = _theta(r)
    ref = _run(d, r, Y, M, C0, x0, init, theta=th, dynamics=1, kernel=1)
    eng = _engine(d, r, init, C0, x0, theta=th, dynamics=3, kernel=1)
    Yd = _padded(Y[None], torch.float64, eng.device)[0]
    Md = _padded(M[None], torch.uint8, eng.device)[0]
    mom = torch.zeros((1, T, so.nmom(r)), dtype=torch.float64, device=eng.device)
    for t in range(T):
        x = eng.get_state(want_C=False)["x"].cpu().numpy()
        arg = 2 * np.pi * th * (t + 1) + x
        eng.run(Yd[:, t:t + 1], Md[:, t:t + 1], k0=t + 1, want_X=False, xbar=np.cos(arg), F=np.diag(-np.sin(arg)),
                moments_out=mom[:, t:t + 1])
        assert eng.status() == -1
    assert eng.launch_info()["kernel"] == "direct"
    assert relerr(mom[0].cpu().numpy(), ref["mom"][0]) < 1e-12
    eng.close()


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("case", ["plain", "loglik", "grad_linear", "eval"])
def test_record_does_not_change_other_outputs(kernel, case):
    """X, Yrec, the scalar record, grad_out, eval, status() and the final state are the same bits with and without a moment
    buffer; a moments-only run writes the 8-wide record; a run after the buffer is cleared gives the bits of a fresh engine."""
    if case == "eval" and kernel == 2:
        pytest.skip("fused evaluation runs on the direct-load and batch kernels")
    r = 8
    d = 960 if kernel != 3 else 203
    Y, M, C0, x0 = _masked(d, r, None, seed=11 + kernel)
    init = _init(r, d, False)
    kw = dict(KERNEL_KW[kernel])
    if case == "loglik":
        kw["loglik"] = True
    if case == "grad_linear":
        A, c = _dynamics(r, 2)
        kw.update(dynamics=2, grad_linear=True, A=A, c=c, want_grad=True)
    if case == "eval":
        E = (np.random.RandomState(4).rand(*Y.shape) < 0.15).astype(np.uint8)
        kw.update(E=E, Yorig=Y + 0.01)
    a = _run(d, r, Y, M, C0, x0, init, moments=True, **kw)
    b = _run(d, r, Y, M, C0, x0, init, moments=False, **kw)
    assert a["info"]["kernel"] == b["info"]["kernel"] == KNAME[kernel]
    for k in ("X", "Yrec", "scal", "status"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    for k in ("grad", "eval"):
        assert all(np.array_equal(u, v) for u, v in zip(a[k], b[k])), k
    for k, v in a["state"].items():
        assert v is None or np.array_equal(v, b["state"][k]), k
    assert a["scal"].shape[-1] == (10 if case == "loglik" else 8)
    # the buffer is cleared after each run: a following run without it gives the bits of a fresh engine
    if case == "plain":
        torch = _torch()
        c = _run(d, r, Y, M, C0, x0, init, moments=True, keep=True, **kw)
        eng = c["engine"]
        eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        Yd = _padded(Y[None], torch.float64, eng.device)[0]
        Md = _padded(M[None], torch.uint8, eng.device)[0]
        X1 = eng.run(Yd[:, :5], Md[:, :5], k0=1, want_X=True)["X"].cpu().numpy()
        X2 = eng.run(Yd[:, 5:], Md[:, 5:], k0=6, want_X=True)["X"].cpu().numpy()
        eng.close()
        assert np.array_equal(np.concatenate([X1, X2])[None], b["X"])


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("r", [5, 16], ids=lambda r: "r%d" % r)
def test_horizon_across_launches_is_bit_identical(kernel, r):
    d = 960 if kernel != 3 else 203
    Y, M, C0, x0 = _masked(d, r, None, seed=17 * r)
    init = _init(r, d, False)
    one = _run(d, r, Y, M, C0, x0, init, chunks=[0, 12], **KERNEL_KW[kernel])
    two = _run(d, r, Y, M, C0, x0, init, chunks=[0, 5, 12], **KERNEL_KW[kernel])
    if kernel == 2:
        # The TMA-staged kernel forms the statistics of step t from C_{t-1} and corrects them algebraically for the pending
        # rank-1 update g_{t-1} (A_t = A0 + u g' + g u' + kappa g g').  At a launch boundary that update is already in C, so the
        # first step of the next launch sums other terms of the same value: the records agree to rounding, not bit for bit.
        assert np.array_equal(one["mom"][:, :5], two["mom"][:, :5])
        assert relerr(two["mom"], one["mom"]) < 1e-12 and relerr(two["Xs"], one["Xs"]) < 1e-12 and relerr(two["Ps"], one["Ps"]) < 1e-12
    else:
        assert np.array_equal(one["mom"], two["mom"]) and np.array_equal(one["Xs"], two["Xs"]) and np.array_equal(one["Ps"], two["Ps"])


@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_external_exchange_records_agree(world):
    """Row-sharded ranks (caller-driven exchange, emulated in one process) write bit-identical records; their smoothed X
    matches a single engine's."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, shard_rows
    r, d = 8, 4001
    Y, M, C0, x0 = _masked(d, r, None, seed=91)
    init = _init(r, d, False)
    splits = [shard_rows(d, world, i) for i in range(world)]
    engs = []
    for i, (b, e) in enumerate(splits):
        eng = FilterEngine(e - b, r, kernel=1, exchange="external", world_size=world, rank=i, d_global=d)
        eng.set_state(C_=C0[b:e], V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        engs.append(eng)
    dev = engs[0].device
    Yd = [torch.as_tensor(np.ascontiguousarray(Y[:, b:e])).to(dev) for b, e in splits]
    Md = [torch.as_tensor(np.ascontiguousarray(M[:, b:e])).to(dev) for b, e in splits]
    moms = [torch.zeros((1, T, so.nmom(r)), dtype=torch.float64, device=dev) for _ in range(world)]
    bufs = [eng.stats_buffer() for eng in engs]
    for t in range(T):
        for i, eng in enumerate(engs):
            eng.run(Yd[i][t:t + 1], Md[i][t:t + 1], k0=1 + t, want_X=False)
        tot = torch.zeros_like(bufs[0])
        for buf in bufs:
            tot += buf
        for buf in bufs:
            buf.copy_(tot)
        for i, eng in enumerate(engs):
            eng.run(Yd[i][t:t + 1], Md[i][t:t + 1], k0=1 + t, want_X=False, moments_out=moms[i][:, t:t + 1], _finish=True)
    for eng in engs:
        assert eng.status() == -1
    ref = _run(d, r, Y, M, C0, x0, init, kernel=1)
    m0 = moms[0].cpu().numpy()
    for i in range(1, world):
        assert np.array_equal(moms[i].cpu().numpy(), m0)
    Xs = engs[0].smooth(moms[0]).cpu().numpy()
    assert relerr(Xs, ref["Xs"][0]) < 1e-9
    for eng in engs:
        eng.close()


def test_refusals():
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    from rpsmf_b200._capi import PsmfError
    r, d = 4, 500
    Y, M, C0, x0 = _masked(d, r, None, seed=2)
    init = _init(r, d, False)
    eng = _engine(d, r, init, C0, x0, simplified=True, kernel=1)
    Yd = torch.as_tensor(Y).to(eng.device)
    with pytest.raises(PsmfError):
        eng.run(Yd, want_moments=True)
    with pytest.raises(PsmfError):
        eng.smooth(torch.zeros((T, so.nmom(r)), dtype=torch.float64, device=eng.device))
    eng.close()
    eng = _engine(d, r, init, np.stack([C0, C0]), np.stack([x0, x0]), S=2, kernel=1)
    L = eng._L
    buf = torch.zeros((2, T, so.nmom(r)), dtype=torch.float64, device=eng.device)
    import ctypes as C
    assert L.psmf_set_moments(eng._h, C.c_void_p(buf.data_ptr()), so.nmom(r) - 1) == -1          # stride below one record
    assert L.psmf_set_moments(eng._h, C.c_void_p(buf.data_ptr()), so.nmom(r)) == 0                # fits one step ...
    Y2 = torch.as_tensor(np.stack([Y, Y])).to(eng.device)
    assert L.psmf_set_moments(eng._h, None, 0) == 0
    xs = torch.empty((2, T, r), dtype=torch.float64, device=eng.device)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert L.psmf_smooth(eng._h, C.c_void_p(buf.data_ptr()), buf.stride(0), 0, C.c_void_p(xs.data_ptr()), None, s) == -1
    assert L.psmf_smooth(eng._h, C.c_void_p(buf.data_ptr()), T, T, C.c_void_p(xs.data_ptr()), None, s) == -1   # series overlap
    with pytest.raises(ValueError):
        eng.run(Y2, moments_out=buf[:, :, 1:])
    eng.close()
    # ... but a run of T steps through a one-step stride is refused at the launch
    eng = _engine(d, r, init, np.stack([C0, C0]), np.stack([x0, x0]), S=2, kernel=1)
    assert eng._L.psmf_set_moments(eng._h, C.c_void_p(buf.data_ptr()), so.nmom(r)) == 0
    from rpsmf_b200 import _capi
    io = _capi.PsmfIO()
    io.Y, io.ldy, io.y_series_stride = Y2.data_ptr(), d, T * d
    assert eng._L.psmf_run(eng._h, C.byref(io), T, 1, s) == -1
    eng._L.psmf_set_moments(eng._h, None, 0)
    eng.close()
    # Q = 0 and P = 0: the filter runs, the smoother meets a singular P_bar
    init0 = dict(init, Q=np.zeros((r, r)), P=np.zeros((r, r)))
    res = _run(d, r, Y, M, C0, x0, init0, keep=True, kernel=1)
    assert res["status"] == [-1, -1]
    with pytest.raises(FloatingPointError):
        res["engine"].smooth(res["mom"])
    res["engine"].close()
    with pytest.raises(ValueError):
        from rpsmf_b200 import rPSMFIter
        rPSMFIter(None, C0, init["V"], x0.reshape(r, 1), init["P"], init["Q"], init["rho"] * np.eye(d), 1.8, None, simplified=True,
                  smooth=True)


@pytest.mark.parametrize("ue", [1, 7])
def test_recursive_classes_join_the_horizon(ue):
    from rpsmf_b200 import rPSMFIter, rPSMFRecursive
    from rpsmf_b200.nonlinearities import RandomWalk
    r, d = 5, 300
    Y, M, C0, x0 = make_problem(d, r, T, seed=8)
    init = _init(r, d, False)
    y = {k + 1: Y[k].reshape(d, 1) for k in range(T)}
    R0 = init["rho"] * np.eye(d)
    mk = lambda cls, **kw: cls(np.zeros(0), C0.copy(), init["V"], x0.reshape(r, 1), init["P"], init["Q"], R0, init["lam"],
                               RandomWalk(), smooth=True, **kw)
    it = mk(rPSMFIter)
    it.optim_init()
    it.step(y, 1, T)
    rec = mk(rPSMFRecursive)
    rec.run(y, T, 0, update_every=ue)
    ref = _oracle_record(Y, None, C0, x0, init, robust=True)
    Xo, Po = so.rts(ref, r)
    for k in range(1, T + 1):
        assert np.array_equal(rec._mu_smooth[k], it._mu_smooth[k]) and np.array_equal(rec._P_smooth[k], it._P_smooth[k])
        assert relerr(rec._mu_smooth[k].reshape(-1), Xo[k - 1]) < TOL and relerr(rec._P_smooth[k], Po[k - 1]) < TOL
    it.close()
    rec.close()


def test_efull_smooth_is_masked_per_series():
    """A series whose smoothed states are not finite (Q = 0, P = 0: P_bar is singular) gets NaN; the others keep their value."""
    torch = _torch()
    from rpsmf_b200.impute import _smoothed_efull
    r, d, S = 4, 300, 3
    Y, M, C0, x0 = _masked(d, r, S, seed=6)
    init = _init(r, d, False)
    eng = _engine(d, r, init, C0, x0, S=S, kernel=1)
    Q = np.stack([init["Q"], np.zeros((r, r)), init["Q"]])
    P = np.stack([init["P"], np.zeros((r, r)), init["P"]])
    eng.set_state(Q=Q, P=P)
    Yd = torch.as_tensor(Y).to(eng.device)
    Md = torch.as_tensor(M).to(eng.device)
    E = torch.as_tensor((np.random.RandomState(1).rand(S, T, d) < 0.2).astype(np.uint8)).to(eng.device)
    out = eng.run(Yd, Md, want_X=False, want_moments=True)
    assert eng.status() == -1
    efs = _smoothed_efull(eng, out["moments"], Yd + 0.5, E)
    assert np.isfinite(efs[0]) and np.isnan(efs[1]) and np.isfinite(efs[2])
    with pytest.raises(FloatingPointError):
        eng.smooth(out["moments"])
    eng.close()


def _pm25():
    from conftest import impute_case, load_golden
    g = load_golden("impute_pm25_30")
    return g, impute_case(g)


@pytest.mark.parametrize("method", ["rPSMF", "PSMF"])
def test_imputation_efull_smooth(method):
    from rpsmf_b200 import ProbabilisticSequentialMatrixFactorizer, robust_PSMF
    from rpsmf_b200.impute import fit_repeats
    torch = _torch()
    g, c = _pm25()
    r = c["r"]
    d, n = c["Y"].shape
    Einit = float(g["rep0_%s_Einit" % method])
    V, Q, R, P = 2 * np.eye(r), 0.1 * np.eye(r), 10 * np.eye(d), np.eye(r)
    args = lambda X: (c["Y"], c["C0"].copy(), X, d, n, r, c["M"], c["Mmiss"])
    if method == "rPSMF":
        f = lambda X, **kw: robust_PSMF(*args(X), V, Q, R, P, 1.8, 2, c["Iter"], c["YorigInt"], Einit, **kw)
    else:
        f = lambda X, **kw: ProbabilisticSequentialMatrixFactorizer(*args(X), 0, V, Q, R, P, 2, c["Iter"], c["YorigInt"], Einit, **kw)
    X1, X2 = c["X0"].copy(), c["X0"].copy()
    plain = f(X1)
    sm = f(X2, smooth=True)
    assert len(plain) == 4 and len(sm) == 5
    assert np.array_equal(plain[0], sm[0]) and np.array_equal(plain[1], sm[1]) and plain[3] == sm[3]   # Epred, Efull, InsideBars
    assert np.array_equal(X1, X2)                          # X is the filtered states either way
    efs = sm[4]
    assert efs.shape == plain[1].shape and efs[0, 0] == Einit
    # numpy: C_T X^s over Mmiss, C_T and the records from a rerun of the engine at the last sweep (fit_repeats, one series)
    Ys, Cs, Xs, Ms, Mm = [c["Y"]], [c["C0"].copy()], [c["X0"].copy()], [c["M"]], [c["Mmiss"]]
    fr = fit_repeats(Ys, Cs, Xs, Ms, Mm, V, Q, R, P, 1.8 if method == "rPSMF" else 0.0, 2, c["Iter"], c["YorigInt"], [Einit],
                     robust=method == "rPSMF", smooth=True)
    frp = fit_repeats(Ys, [c["C0"].copy()], [c["X0"].copy()], Ms, Mm, V, Q, R, P, 1.8 if method == "rPSMF" else 0.0, 2, c["Iter"],
                      c["YorigInt"], [Einit], robust=method == "rPSMF")
    assert np.array_equal(fr[0][0], frp[0][0]) and np.array_equal(fr[1][0], frp[1][0]) and fr[3] == frp[3]
    assert relerr(fr[4][0], efs) < 1e-9
    # EfullSmooth against numpy on an engine run of the same sweeps
    from rpsmf_b200 import FilterEngine
    from rpsmf_b200.engine import ingest, transpose_mask
    robust = method == "rPSMF"
    eng = FilterEngine(d, r, robust=robust, c_update_transpose=robust)
    Yt, _ = ingest(c["Y"])
    Mt = transpose_mask(c["M"])
    eng.set_state(C_=c["C0"], V=V, P=P, x=np.ascontiguousarray(c["X0"][:, n - 1]), Q=Q, rho=[10.0], lam=[1.8 if robust else 0.0])
    for i in range(c["Iter"]):
        if robust:
            eng.set_state(Q=Q, rho=[10.0], lam=[1.8])
        out = eng.run(Yt, Mt, k0=1, want_X=True, want_moments=True)
        Xsm = eng.smooth(out["moments"]).cpu().numpy()
        CT = eng.get_state()["C"].cpu().numpy()
        Yhat = CT @ Xsm.T
        Mmiss = c["Mmiss"] != 0
        ref = np.sqrt(np.sum((Yhat - c["YorigInt"])[Mmiss] ** 2) / np.sum(Mmiss))
        assert abs(efs[0, i + 1] - ref) / ref < 1e-9
    eng.close()


def test_row_sharded_ranks_share_one_gpu():
    """Two row-sharded ranks on cuda:0 exchanging through the in-kernel NVLink mailboxes (tests/multi_gpu_smooth_check.py):
    the moment records are bit-identical on both ranks and the smoothed X is within 1e-9 of the one-GPU engine's, on the
    direct-load and the TMA-staged kernel."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29524", os.path.join(root, "tests", "multi_gpu_smooth_check.py"), "--same-device"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, PSMF_SPIN_TIMEOUT_MS="60000"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" OK") == 4 and "FAIL" not in r.stdout
