"""Every filter kernel variant, at every latent rank and both storage types, against the float64 oracle.

The library compiles each kernel once per rank r = 1..16 and per storage type, and much of its code depends on r (the
single-block Gram at r <= 8 against the split form, the paired tiles of the batch kernel, the Gauss-Jordan result buffer
picked by r & 1, the chunk size of the TMA-staged kernel).  Automatic dispatch sends most small test shapes to the
batch kernel, so every case here forces its kernel and then checks from launch_info() that the variant it meant to
test is the one that ran: a case that lands elsewhere fails.

Tolerances follow the rest of the suite: fp64 1e-9 norm-wise per quantity, fp32 storage 1e-4 against the oracle run
on fp32-rounded Y and C0; masks, counts and memory a kernel must not touch are compared exactly.
"""

import numpy as np
import pytest

from conftest import relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem
from test_gpu_filter import TOL, _compare, _engine_run, _oracle_run, _torch

pytestmark = pytest.mark.gpu

TOL32 = 1e-4
RANKS = list(range(1, 17))
SPLIT_RANKS = [5, 8, 9, 16]        # both sides of the r <= 8 Gram split, odd and even r (Gauss-Jordan result buffer)
T = 12
CHUNKS = [0, 5, 12]                # two launches: the pending rank-1 update is flushed at the launch boundary
KNAME = {1: "direct", 2: "tma", 3: "batch"}


def _sms():
    return _torch().cuda.get_device_properties(0).multi_processor_count


def _v2_ts(r, esize):
    """Tiles per chunk slot of the TMA-staged kernel (v2_ts in psmf_common.cuh)."""
    return max(4, min(16, 16384 // (r * 32 * esize)))


def _tma_plan(r, esize, ntiles, static_smem, max_smem=232448):
    """(nslot, nchunks) of a one-CTA TMA-staged launch, as psmf_create sizes it (psmf_capi.cu): chunk slots of v2_ts tiles
    fill the shared memory (227 KB opt-in on a B200) left by the static part and the residual buffer."""
    ts = _v2_ts(r, esize)
    slot = (ts * r * 32 * esize + 127) // 128 * 128
    nchunks = -(-ntiles // ts)
    avail = max_smem - static_smem - ntiles * 32 * 8 - 256
    return (min(avail // slot, nchunks, 64) if avail > 0 else 0), nchunks


def _stream_d(r, esize):
    """A row count whose one-CTA TMA launch streams: more chunks than slots, and at least the 5 slots a ring needs.
    The static shared memory of the kernel is not known here; the middle of the band that works for anything from 0
    to 40 KB is taken, and the test checks the outcome through launch_info()."""
    def streams(n):
        for static in (0, 40000):
            nslot, nchunks = _tma_plan(r, esize, n, static)
            if not (5 <= nslot < nchunks):
                return False
        return True
    good = [n for n in range(2, 2000) if streams(n)]
    return 32 * ((good[0] + good[-1]) // 2)


# variant -> (kernel, d, S, engine keywords); d is a function of (r, esize) for the streaming TMA variant
VARIANTS = {
    "direct": (1, 4001, None, {}),                   # 126 tiles, 7 CTAs (cooperative grid reduce), last tile holds one row
    "direct_S3": (1, 4001, 3, {}),                   # one CTA per series, per-series state / output offsets
    "rhovec": (1, 4001, None, dict(rho_vector=True)),
    "rhovec_S3": (1, 4001, 3, dict(rho_vector=True)),
    "tma_resident": (2, 1600, None, dict(ctas=2)),
    "tma_stream": (2, _stream_d, None, dict(ctas=1)),
    "batch8": (3, 1100, 3, {}),                      # 35 tiles: tiles 32..34 are read without the prefetch
    "batch4": (3, 203, 3, {}),                       # 7 tiles: fewer than 8 -> the 4-warp form
}


def _check_variant(name, info, r, esize, d):
    """Section 1 of the matrix: the kernel that ran is the variant the case is about."""
    kernel = VARIANTS[name][0] if name in VARIANTS else 3
    assert info["kernel"] == KNAME[kernel], (name, info)
    if name == "direct" or name == "rhovec":
        assert info["ctas"] > 1, info
    if name == "tma_resident":
        assert info["resident"] is True, info
    if name == "tma_stream":
        ts = _v2_ts(r, esize)
        nchunks = -(-((d + 31) // 32) // ts)
        assert info["resident"] is False and info["nslot"] >= 5 and nchunks > info["nslot"], (info, nchunks)
    if name == "batch8":
        assert info["threads"] == 256, info
    if name in ("batch4", "batch4_many"):
        assert info["threads"] == 128, info


def _dtype(tag):
    torch = _torch()
    return (torch.float64, 8, TOL) if tag == "f64" else (torch.float32, 4, TOL32)


def _rounded(a, tag):
    return a if tag == "f64" else a.astype(np.float32).astype(np.float64)


def _series(res, s):
    X, Yrec, scal, st, info = res
    return X[s], Yrec[s], scal[s], {k: (v[s] if v is not None and np.ndim(v) > 0 else v) for k, v in st.items()}, info


def _compare_all(res, Y, M, C0, x0, init, cfg, S, tag, tol):
    """Every series against the oracle (on the fp32-rounded Y and C0 for fp32 storage)."""
    rho = init["rho"]
    for s in range(S or 1):
        one = (lambda a: a) if S is None else (lambda a: a[s])
        ref = _oracle_run(_rounded(one(Y), tag), one(M), _rounded(one(C0), tag), one(x0), init, cfg)
        got = res if S is None else _series(res, s)
        if np.ndim(rho) > 0:
            # a non-uniform diagonal R is kept as the caller's vector times a scale, and the scalar record holds the scale
            ost, oX, oYrec, oscal = ref
            oscal = oscal.copy()
            oscal[:, 7] /= np.mean(rho)
            ref = (ost, oX, oYrec, oscal)
        _compare(got, ref, tol)


def _masked_problem(d, r, S, seed):
    """A masked problem with rows that are never observed (their C rows must come back bit for bit)."""
    Y, M, C0, x0 = make_problem(d, r, T, seed=seed, S=S)
    dead = np.array([1, d // 2])
    M[..., dead] = 0
    Y = Y * M
    return Y, M, C0, x0, dead


def _init(r, d, rho_vector, seed=0):
    init = impute_init(r)
    if rho_vector:
        init["rho"] = 10.0 * (0.5 + np.random.RandomState(seed).rand(d))      # distinct rho_i
    return init


def _matrix_cell(name, r, tag, kernel, d, S, kw):
    dtype, esize, tol = _dtype(tag)
    rho_vector = kw.get("rho_vector", False)
    Y, M, C0, x0, dead = _masked_problem(d, r, S, seed=100 * r + d % 97)
    init = _init(r, d, rho_vector)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, dtype=dtype, chunks=CHUNKS, S=S, kernel=kernel, **kw)
    _check_variant(name, res[4], r, esize, d)
    _compare_all(res, Y, M, C0, x0, init, po.OracleConfig(robust=True), S, tag, tol)
    # never-observed rows keep their C row bit for bit
    C = res[3]["C"]
    assert np.array_equal(C[..., dead, :], _rounded(C0, tag)[..., dead, :])
    # a step with every row missing is a pure prediction step: finite, and x does not move under identity dynamics
    Yz, Mz = Y[..., :4, :].copy(), M[..., :4, :].copy()
    Mz[..., 2, :] = 0
    Yz = Yz * Mz
    X, Yrec, scal, st, info = _engine_run(d, r, Yz, Mz, C0, x0, init, True, dtype=dtype, S=S, kernel=kernel, **kw)
    assert info["kernel"] == KNAME[kernel]
    assert np.isfinite(X).all() and np.isfinite(Yrec).all() and np.isfinite(scal).all()
    assert all(np.isfinite(v).all() for v in st.values() if v is not None)
    assert np.array_equal(X[..., 2, :], X[..., 1, :])


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", RANKS, ids=lambda r: "r%d" % r)
@pytest.mark.parametrize("name", list(VARIANTS))
def test_rank_matrix(name, r, tag):
    kernel, d, S, kw = VARIANTS[name]
    if callable(d):
        d = d(r, _dtype(tag)[1])
    _matrix_cell(name, r, tag, kernel, d, S, kw)


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("r", [1, 8, 9, 16], ids=lambda r: "r%d" % r)
def test_rank_matrix_batch4_past_prefetch(r, tag):
    """More than 2 series per SM select the 4-warp batch kernel; 19 tiles per series take it past its 16 prefetched
    tiles (V3_PF per warp)."""
    _matrix_cell("batch4_many", r, tag, 3, 600, 2 * _sms() + 1, {})


# ---- flags and dynamics on each kernel -------------------------------------------------------------------------------
# One shape every kernel accepts: d = 960 (30 tiles, d % 16 == 0).  Direct: 3 CTAs; TMA: 2 data CTAs, resident; batch:
# one series, 8 warps.
FLAG_D = 960
KERNEL_KW = {1: dict(kernel=1, ctas=3), 2: dict(kernel=2, ctas=2), 3: dict(kernel=3)}


def _theta(r):
    return 0.05 + 0.1 * np.random.RandomState(r).rand(r)


FLAG_CASES = {
    # id: (engine keywords, oracle keywords, dynamics cos)
    "psmf_vt": (dict(robust=False, c_update_transpose=True), dict(robust=False, c_update_transpose=True), False),
    "psmf_vtt": (dict(robust=False, c_update_transpose=False), dict(robust=False, c_update_transpose=False), False),
    "fixed_lambda": (dict(robust=True, fixed_lambda=True), dict(robust=True, fixed_lambda=True), False),
    "alpha_beta": (dict(robust=True, alpha=0.97, beta=1.06), dict(robust=True, alpha=0.97, beta=1.06), False),
    "simplified_cos": (dict(robust=True, simplified=True), dict(robust=True, simplified=True), True),
    "simplified_cos_psmf": (dict(robust=False, simplified=True), dict(robust=False, simplified=True), True),
    "cos": (dict(robust=True), dict(robust=True), True),
}

FLAG_PARAMS = [(c, k, r, "f64") for c in FLAG_CASES for k in (1, 2, 3) for r in SPLIT_RANKS] + \
              [(c, k, 9, "f32") for c in FLAG_CASES for k in (1, 2, 3)]


@pytest.mark.parametrize("case,kernel,r,tag", FLAG_PARAMS,
                         ids=["%s-%s-r%d-%s" % (c, KNAME[k], r, t) for c, k, r, t in FLAG_PARAMS])
def test_flags_on_each_kernel(case, kernel, r, tag):
    from rpsmf_b200 import _capi
    ekw, okw, cos = FLAG_CASES[case]
    dtype, esize, tol = _dtype(tag)
    d = FLAG_D
    Y, M, C0, x0, dead = _masked_problem(d, r, None, seed=7 * r + kernel)
    init = impute_init(r)
    ekw = dict(ekw)
    robust = ekw.pop("robust")
    if cos:
        init["theta"] = _theta(r)
        ekw["dynamics"] = _capi.DYN_COS
        okw = dict(okw, dynamics=po.DYN_COS)
    res = _engine_run(d, r, Y, M, C0, x0, init, robust, dtype=dtype, chunks=CHUNKS, **KERNEL_KW[kernel], **ekw)
    assert res[4]["kernel"] == KNAME[kernel]
    _compare_all(res, Y, M, C0, x0, init, po.OracleConfig(**okw), None, tag, tol)
    assert np.array_equal(res[3]["C"][dead], _rounded(C0, tag)[dead])


def _grad_reference(Y, M, C0, x0, init, ll_student, d):
    """Summed theta gradient of the step log-likelihood under cos dynamics, from the oracle's trajectory: every step uses
    the C, V and lambda entering it and its own eta.  With a mask the likelihood is restated over the observed rows
    (n = n_obs, q = sum of e^2 over observed rows, C'Me), the form the kernels implement (psmf_filter.cuh, small_update).
    The reference defines the gradient for complete data only (psmf.py:48-66), so this masked form is pinned against
    nothing but this restatement."""
    cfg = po.OracleConfig(robust=True, dynamics=po.DYN_COS)
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"],
                        init["lam"], init["theta"])
    grad = np.zeros_like(x0)
    for t in range(Y.shape[0]):
        k = 1 + t
        m = np.ones(d) if M is None else M[t].astype(float)
        new, out = po.step(st, cfg, Y[t], m, k=k)
        if M is None:
            grad += po.theta_grad_cos(ll_student, st.theta, st.x, k, Y[t], st.C, st.V, out["eta"], st.lam, d)
        else:
            arg = 2.0 * np.pi * st.theta * k + st.x
            f = np.cos(arg)
            e = m * (Y[t] - st.C @ f)
            g_f = po.dll_df(ll_student, f, st.V, st.C.T @ e, float(e @ e), out["eta"], st.lam, float(m.sum()))
            grad += g_f * (-np.sin(arg)) * (2.0 * np.pi * k)
        st = new
    return grad


GRAD_PARAMS = [(k, r, s) for k in (1, 2, 3) for r in SPLIT_RANKS for s in (False, True)]


@pytest.mark.parametrize("kernel,r,ll_student", GRAD_PARAMS,
                         ids=["%s-r%d-%s" % (KNAME[k], r, "student" if s else "gauss") for k, r, s in GRAD_PARAMS])
def test_theta_gradient_unmasked(kernel, r, ll_student):
    from rpsmf_b200 import _capi
    d = FLAG_D
    Y, _, C0, x0 = make_problem(d, r, T, seed=40 + r, missing=0.0)
    init = impute_init(r)
    init["theta"] = _theta(r)
    res = _engine_run(d, r, Y, None, C0, x0, init, True, chunks=CHUNKS, want_grad=True, dynamics=_capi.DYN_COS,
                      ll_student=ll_student, **KERNEL_KW[kernel])
    assert res[4]["kernel"] == KNAME[kernel]
    _compare(res, _oracle_run(Y, None, C0, x0, init, po.OracleConfig(robust=True, dynamics=po.DYN_COS)), TOL)
    ref = _grad_reference(Y, None, C0, x0, init, ll_student, d)
    assert relerr(res[3]["grad"], ref) < TOL


@pytest.mark.parametrize("r", SPLIT_RANKS)
@pytest.mark.parametrize("ll_student", [False, True], ids=["gauss", "student"])
def test_theta_gradient_masked_kernels_agree(r, ll_student):
    from rpsmf_b200 import _capi
    d = FLAG_D
    Y, M, C0, x0, _ = _masked_problem(d, r, None, seed=60 + r)
    init = impute_init(r)
    init["theta"] = _theta(r)
    grads = []
    for kernel in (1, 2, 3):
        res = _engine_run(d, r, Y, M, C0, x0, init, True, chunks=CHUNKS, want_grad=True, dynamics=_capi.DYN_COS,
                          ll_student=ll_student, **KERNEL_KW[kernel])
        assert res[4]["kernel"] == KNAME[kernel]
        grads.append(res[3]["grad"])
    assert relerr(grads[1], grads[0]) < 1e-11 and relerr(grads[2], grads[0]) < 1e-11
    assert relerr(grads[0], _grad_reference(Y, M, C0, x0, init, ll_student, d)) < TOL


@pytest.mark.parametrize("kernel", [1, 2, 3], ids=lambda k: KNAME[k])
@pytest.mark.parametrize("r", SPLIT_RANKS)
def test_nan_mask_bit_identical(kernel, r):
    d = FLAG_D
    Y, M, C0, x0, _ = _masked_problem(d, r, None, seed=80 + r)
    init = impute_init(r)
    a = _engine_run(d, r, Y, M, C0, x0, init, True, chunks=CHUNKS, **KERNEL_KW[kernel])
    Yn = Y.copy()
    Yn[M == 0] = np.nan
    b = _engine_run(d, r, Yn, None, C0, x0, init, True, chunks=CHUNKS, nan_mask=True, **KERNEL_KW[kernel])
    assert a[4]["kernel"] == b[4]["kernel"] == KNAME[kernel]
    for i in range(3):
        assert np.array_equal(a[i], b[i])
    assert np.array_equal(a[3]["C"], b[3]["C"]) and np.array_equal(a[3]["V"], b[3]["V"])


# ---- layouts: inputs and outputs inside larger buffers ---------------------------------------------------------------
LAYOUTS = [
    # kernel, d, S, row padding of Y / M (/ Yorig / E), gap between series, row padding of Yrec, fused evaluation
    (1, 4001, 3, 3, 7, 5, True),
    (3, 1100, 3, 3, 7, 5, True),
    (2, 1600, None, 16, 0, 16, False),      # bulk copies: rows of Y and M stay 16-byte aligned
]
LAYOUT_PARAMS = [(lay, r, tag) for lay in LAYOUTS for r in (5, 16) for tag in ("f64", "f32")]


@pytest.mark.parametrize("layout,r,tag", LAYOUT_PARAMS,
                         ids=["%s-r%d-%s" % (KNAME[lay[0]], r, t) for lay, r, t in LAYOUT_PARAMS])
def test_strided_layouts_bit_identical(layout, r, tag):
    kernel, d, S, pad, gap, rec_pad, fused = layout
    dtype = _dtype(tag)[0]
    Y, M, C0, x0, _ = _masked_problem(d, r, S, seed=90 + r)
    init = impute_init(r)
    kw = dict(kernel=kernel, dtype=dtype, chunks=CHUNKS, S=S)
    if fused:
        rng = np.random.RandomState(r)
        Yorig = Y + rng.randn(*Y.shape)
        E = ((rng.rand(*Y.shape) < 0.1) & (M == 0)).astype(np.uint8)
        kw.update(Yorig=Yorig, E=E)
    a = _engine_run(d, r, Y, M, C0, x0, init, True, **kw)
    b = _engine_run(d, r, Y, M, C0, x0, init, True, pad=pad, gap=gap, rec_pad=rec_pad, **kw)
    assert a[4]["kernel"] == b[4]["kernel"] == KNAME[kernel]
    for i in range(3):
        assert np.array_equal(a[i], b[i])
    for k in ("C", "V", "P", "x", "rho", "lam") + (("eval",) if fused else ()):
        assert np.array_equal(a[3][k], b[3][k]), k
    if fused:
        assert a[3]["eval"][..., 2].sum() == E.sum()          # every marked entry counted once


def _fresh_run(d, r, Y, M, C0, x0, init, eng=None, **kw):
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    if eng is None:
        eng = FilterEngine(d, r, robust=True, **kw)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    out = eng.run(torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda(), want_X=True)
    assert eng.status() == -1
    X = out["X"].cpu().numpy()
    C = eng.get_state()["C"].cpu().numpy()
    return X, C, eng.launch_info()


def test_misaligned_input_leaves_the_tma_kernel():
    """Y one element off 16-byte alignment: automatic dispatch falls back to the direct-load kernel with the same
    result to rounding; forcing the TMA-staged kernel is an error, after which the engine still runs aligned input
    exactly as a fresh engine does."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r = 1600, 16
    Y, M, C0, x0, _ = _masked_problem(d, r, None, seed=5)
    init = impute_init(r)
    Xa, Ca, info = _fresh_run(d, r, Y, M, C0, x0, init, kernel=0)
    assert info["kernel"] == "tma"
    buf = torch.empty(T * d + 1, dtype=torch.float64, device="cuda")
    Yoff = buf[1:].view(T, d)
    Yoff.copy_(torch.as_tensor(Y))
    Md = torch.as_tensor(M).cuda()
    eng = FilterEngine(d, r, robust=True, kernel=0)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Xo = eng.run(Yoff, Md, want_X=True)["X"].cpu().numpy()
    assert eng.status() == -1 and eng.launch_info()["kernel"] == "direct"
    assert relerr(Xo, Xa) < 1e-12 and relerr(eng.get_state()["C"].cpu().numpy(), Ca) < 1e-12
    eng.close()
    eng = FilterEngine(d, r, robust=True, kernel=2)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    with pytest.raises(_capi.PsmfError):
        eng.run(Yoff, Md, want_X=True)
    Xb, Cb, info = _fresh_run(d, r, Y, M, C0, x0, init, eng=eng)
    assert info["kernel"] == "tma"
    assert np.array_equal(Xb, Xa) and np.array_equal(Cb, Ca)
    eng.close()


# ---- eligibility: what the ABI documents as unavailable is refused ---------------------------------------------------
REFUSED_AT_CREATE = {
    "rhovec_tma": dict(d=960, r=8, rho_vector=True, kernel=2),
    "rhovec_batch": dict(d=960, r=8, rho_vector=True, kernel=3),
    "tma_d_not_16": dict(d=1000, r=8, kernel=2),
    "tma_series": dict(d=960, r=8, kernel=2, n_series=2),
    "batch_too_large": dict(d=20000, r=16, kernel=3),
}


@pytest.mark.parametrize("case", list(REFUSED_AT_CREATE))
def test_forced_kernel_refused_at_create(case):
    from rpsmf_b200 import FilterEngine, _capi
    kw = dict(REFUSED_AT_CREATE[case])
    with pytest.raises(_capi.PsmfError):
        FilterEngine(kw.pop("d"), kw.pop("r"), **kw)


def test_forced_tma_refused_at_run_then_engine_still_exact():
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r = FLAG_D, 9
    Y, M, C0, x0, _ = _masked_problem(d, r, None, seed=3)
    init = impute_init(r)
    ref = _fresh_run(d, r, Y, M, C0, x0, init, kernel=2)
    assert ref[2]["kernel"] == "tma"
    eng = FilterEngine(d, r, robust=True, kernel=2)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd, Md = torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda()
    with pytest.raises(_capi.PsmfError):                                     # fused evaluation: direct / batch only
        eng.run(Yd, Md, Yorig=Yd, E=Md)
    X, C, info = _fresh_run(d, r, Y, M, C0, x0, init, eng=eng)
    assert info["kernel"] == "tma" and np.array_equal(X, ref[0]) and np.array_equal(C, ref[1])
    eng.close()
    eng = FilterEngine(d, r, robust=True, kernel=2, dynamics=_capi.DYN_EXTERNAL)
    with pytest.raises(_capi.PsmfError):
        eng.run(Yd[:1], Md[:1], xbar=np.zeros(r), F=np.eye(r))
    eng.close()


@pytest.mark.parametrize("d,kernel", [(1024, "batch"), (1040, "tma"), (1041, "direct")])
def test_auto_dispatch_boundaries(d, kernel):
    """One series: up to 32 tiles the batch kernel; 33 tiles the TMA-staged kernel when d % 16 == 0, else direct."""
    r = 8
    Y, M, C0, x0, _ = _masked_problem(d, r, None, seed=d)
    init = impute_init(r)
    res = _engine_run(d, r, Y, M, C0, x0, init, True)
    assert res[4]["kernel"] == kernel
    _compare(res, _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True)), TOL)
