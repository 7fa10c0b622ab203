"""GPU parity tests: the CUDA filter (through the C ABI) against the oracle and the golden fixtures.

Tolerances: fp64 1e-9 norm-wise per quantity (max|delta| / max|ref|), fp32 storage 1e-4
(BASELINE.json north_star); integer mask handling is exercised through exact zero / non-zero
patterns (a missing row must not move C when y is zero-filled).
"""

import numpy as np
import pytest

from conftest import impute_case, load_golden, relerr
from oracle import psmf_oracle as po
from synth import impute_init, make_problem

pytestmark = pytest.mark.gpu

TOL = 1e-9


def _torch():
    import torch
    return torch


def _padded(a, dtype, dev, pad=0, gap=0, fill=0):
    """(S, T, d) device view of host array `a` inside a larger buffer filled with `fill`: rows of d + pad elements and
    `gap` more elements between series.  Returns (view, buffer)."""
    torch = _torch()
    S, T, d = a.shape
    ld = d + pad
    sst = T * ld + gap
    buf = torch.full((S * sst,), fill, dtype=dtype, device=dev)
    view = buf.as_strided((S, T, d), (sst, ld, 1))
    view.copy_(torch.as_tensor(a).to(dtype))
    return view, buf


def _engine_run(d, r, Y, M, C0, x0, init, robust, ctas=0, dtype=None, chunks=None, S=None, pad=0, gap=0, rec_pad=0,
                want_grad=False, Yorig=None, E=None, sig=2.0, **kw):
    """Run the engine over Y (T, d), or (S, T, d) with S series, in the launches given by `chunks`.  `pad` / `gap` put Y, M
    (and Yorig, E) inside larger buffers (rows of d + pad elements, gaps between series); `rec_pad` writes Yrec into rows
    of d + rec_pad elements whose padding is NaN and must stay so.  Returns (X, Yrec, scal, state, launch_info); with S
    the arrays keep the series axis, the state holds the theta gradient ("grad", summed over the launches) when
    `want_grad` and the fused evaluation sums ("eval", coverage of yhat -+ sig sqrt(U)) when E is given."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    dtype = dtype or torch.float64
    eng = FilterEngine(d, r, dtype=dtype, robust=robust, ctas=ctas, n_series=S or 1, **kw)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=np.atleast_1d(init["rho"]), lam=[init["lam"]],
                  theta=init.get("theta"))
    dev = eng.device
    one = S is None
    Y3 = Y[None] if one else Y
    Yd, _ = _padded(Y3, dtype, dev, pad, gap, float("nan"))
    Md = None if M is None else _padded(M[None] if one else M, torch.uint8, dev, pad, gap, 1)[0]
    Yod = None if Yorig is None else _padded(Yorig[None] if one else Yorig, dtype, dev, pad, gap, float("nan"))[0]
    Ed = None if E is None else _padded(E[None] if one else E, torch.uint8, dev, pad, gap, 1)[0]
    Sn, T = Y3.shape[0], Y3.shape[1]
    Yrec, rec_buf = _padded(np.zeros((Sn, T, d)), dtype, dev, rec_pad, gap if rec_pad else 0, float("nan"))
    bounds = [0, T] if chunks is None else chunks
    Xs, Sc, grad, ev = [], [], 0.0, 0.0
    for a, b in zip(bounds[:-1], bounds[1:]):
        out = eng.run(Yd[:, a:b], None if Md is None else Md[:, a:b], k0=1 + a, want_X=True, Yrec_out=Yrec[:, a:b],
                      want_scal=True, want_grad=want_grad, Yorig=None if Yod is None else Yod[:, a:b],
                      E=None if Ed is None else Ed[:, a:b], sig=sig)
        assert eng.status() == -1
        Xs.append(out["X"].reshape(Sn, b - a, r).cpu().numpy()); Sc.append(out["scal"].reshape(Sn, b - a, -1).cpu().numpy())
        if want_grad:
            grad = grad + out["grad"].cpu().numpy()
        if E is not None:
            ev = ev + out["eval"].cpu().numpy()
    st = {k: (v.double().cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()}
    if want_grad:
        st["grad"] = grad
    if E is not None:
        st["eval"] = ev
    info = eng.launch_info()
    eng.close()
    # the rows of Yrec were written, nothing around them
    keep = torch.ones_like(rec_buf, dtype=torch.bool)
    keep.as_strided(Yrec.shape, Yrec.stride()).fill_(False)
    assert bool(rec_buf[keep].isnan().all())
    X, Yr, Sc = np.concatenate(Xs, axis=1), Yrec.double().cpu().numpy(), np.concatenate(Sc, axis=1)
    if one:
        X, Yr, Sc = X[0], Yr[0], Sc[0]
    return X, Yr, Sc, st, info


def _oracle_run(Y, M, C0, x0, init, cfg, k0=1, record=None):
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"],
                        init["lam"], init.get("theta"))
    return po.run(st, cfg, Y, None if M is None else M.astype(float), k0=k0, record=record)


def _compare(res, ref, tol):
    X, Yrec, scal, st, _ = res
    ost, oX, oYrec, oscal = ref
    assert relerr(X, oX) < tol
    assert relerr(Yrec, oYrec) < tol
    for k in range(8):
        assert relerr(scal[:, k], oscal[:, k]) < tol, po.SCALAR_NAMES[k]
    assert relerr(st["C"], ost.C) < tol
    assert relerr(st["P"], ost.P) < tol
    assert relerr(st["V"], ost.V) < tol
    assert relerr(st["Q"], ost.Q) < tol
    assert relerr(st["x"], ost.x) < tol
    assert relerr(st["rho"], ost.rho) < tol
    assert relerr(st["lam"], ost.lam) < tol


@pytest.mark.parametrize("r", [1, 2, 3, 6, 7, 8, 10, 11, 13, 16])
@pytest.mark.parametrize("robust", [True, False])
def test_ranks_masked(r, robust):
    d, T = 203, 40
    Y, M, C0, x0 = make_problem(d, r, T, seed=r)
    init = impute_init(r)
    cfg = po.OracleConfig(robust=robust, c_update_transpose=robust)
    res = _engine_run(d, r, Y, M, C0, x0, init, robust, c_update_transpose=robust)
    _compare(res, _oracle_run(Y, M, C0, x0, init, cfg), TOL)


@pytest.mark.parametrize("d,ctas", [(5, 0), (32, 0), (33, 1), (1000, 0), (1000, 3), (5000, 0), (5000, 37), (20011, 0)])
def test_shapes_and_grids(d, ctas):
    r, T = 16, 25
    Y, M, C0, x0 = make_problem(d, r, T, seed=d)
    init = impute_init(r)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, ctas=ctas)
    _compare(res, _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True)), TOL)
    if ctas:
        assert res[4]["ctas"] == min(ctas, (d + 31) // 32)


@pytest.mark.parametrize("d,ctas,r,resident", [
    (3840, 1, 16, False),      # one CTA, 20 chunks through a ring of slots (streaming)
    (3856, 1, 16, False),      # last tile half-filled (d % 32 == 16)
    (3840, 3, 16, None),
    (1600, 2, 16, True),       # everything fits the slots: C stays in shared memory
    (20000, 0, 16, None),
    (60000, 0, 16, None),
    (9600, 1, 8, None),
    (9600, 2, 10, None),
    (4800, 1, 3, None),
    (12000, 0, 12, None),
    (300000, 0, 16, False),    # full grid (one data CTA per SM), every CTA streams its chunks through the ring
])
def test_tma_kernel(d, ctas, r, resident):
    T = 12
    Y, M, C0, x0 = make_problem(d, r, T, seed=d + r)
    init = impute_init(r)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, ctas=ctas, kernel=2)
    assert res[4]["kernel"] == "tma"
    if resident is not None:
        assert res[4]["resident"] == resident
    _compare(res, _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True)), TOL)


def test_tma_kernel_variants():
    torch = _torch()
    d, r, T = 7680, 16, 14
    Y, M, C0, x0 = make_problem(d, r, T, seed=77)
    init = impute_init(r)
    ref = _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True))
    # several launches: the pending rank-1 update is flushed at the end of every launch
    res = _engine_run(d, r, Y, M, C0, x0, init, True, ctas=2, kernel=2, chunks=[0, 1, 5, 14])
    assert res[4]["kernel"] == "tma"
    _compare(res, ref, TOL)
    # no mask pointer
    Yf, _, _, _ = make_problem(d, r, T, seed=77, missing=0.0)
    res = _engine_run(d, r, Yf, None, C0, x0, init, True, ctas=2, kernel=2)
    _compare(res, _oracle_run(Yf, None, C0, x0, init, po.OracleConfig(robust=True)), TOL)
    # PSMF (non-robust) and fp32 storage
    res = _engine_run(d, r, Y, M, C0, x0, init, False, ctas=2, kernel=2, c_update_transpose=False)
    _compare(res, _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=False, c_update_transpose=False)), TOL)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, ctas=2, kernel=2, dtype=torch.float32)
    ref32 = _oracle_run(Y.astype(np.float32).astype(np.float64), M, C0.astype(np.float32).astype(np.float64), x0, init,
                        po.OracleConfig(robust=True))
    _compare(res, ref32, 1e-4)
    # both kernels agree to rounding
    a = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=1)
    b = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=2)
    assert a[4]["kernel"] == "direct" and b[4]["kernel"] == "tma"
    assert relerr(a[0], b[0]) < 1e-12 and relerr(a[3]["C"], b[3]["C"]) < 1e-12


@pytest.mark.parametrize("dtype,tol", [("f64", TOL), ("f32", 1e-4)])
def test_resident_regime_at_the_eight_gpu_shard_shape(dtype, tol):
    """The shard one GPU holds when workload L is split over 8 GPUs (125,024 rows, r = 16): full grid, C resident in shared
    memory for the whole launch -- a tile is only handed between producer and pass warps at the initial load and the final
    store.  Several launches (1, 2 and 37 steps: the one- and two-step launches never reach the steady state of the
    pipeline), against the oracle and bit-identical when replayed."""
    torch = _torch()
    d, r, T = 125_024, 16, 40
    Y, M, C0, x0 = make_problem(d, r, T, seed=8)
    init = impute_init(r)
    td = torch.float64 if dtype == "f64" else torch.float32
    res = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=2, dtype=td, chunks=[0, 1, 3, 40])
    assert res[4]["kernel"] == "tma" and res[4]["resident"] and res[4]["ctas"] >= 100
    if dtype == "f64":
        ref = _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True))
    else:
        ref = _oracle_run(Y.astype(np.float32).astype(np.float64), M, C0.astype(np.float32).astype(np.float64), x0, init,
                          po.OracleConfig(robust=True))
    _compare(res, ref, tol)
    again = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=2, dtype=td, chunks=[0, 1, 3, 40])
    assert np.array_equal(res[0], again[0]) and np.array_equal(res[3]["C"], again[3]["C"])
    one = _engine_run(d, r, Y, M, C0, x0, init, True, kernel=2, dtype=td)
    # a launch boundary flushes the pending rank-1 update instead of folding it into the next pass: same values to rounding
    lim = 1e-11 if dtype == "f64" else 1e-5
    assert relerr(one[0], res[0]) < lim and relerr(one[3]["C"], res[3]["C"]) < lim


def test_unmasked_and_all_missing_steps():
    d, r, T = 300, 10, 30
    Y, M, C0, x0 = make_problem(d, r, T, seed=3)
    init = impute_init(r)
    # mask pointer NULL == all observed
    Yfull, _, _, _ = make_problem(d, r, T, seed=3, missing=0.0)
    res = _engine_run(d, r, Yfull, None, C0, x0, init, True)
    _compare(res, _oracle_run(Yfull, None, C0, x0, init, po.OracleConfig(robust=True)), TOL)
    # rows that are always missing, and steps with a single observed row
    M2 = M.copy(); M2[5] = 0; M2[5, 3] = 1; M2[17] = 0; M2[17, 298] = 1; M2[:, 7] = 0; M2[:, 299] = 0
    Y2 = Y * M2
    res = _engine_run(d, r, Y2, M2, C0, x0, init, True)
    _compare(res, _oracle_run(Y2, M2, C0, x0, init, po.OracleConfig(robust=True)), TOL)
    # exactness of the mask handling: a never-observed, zero-filled row of C must not move at all
    assert np.array_equal(res[3]["C"][7], C0[7]) and np.array_equal(res[3]["C"][299], C0[299])


def test_all_rows_missing_step_stays_finite():
    """The reference yields NaN on a step with every row missing (0 * inf at rPSMF.py:113-114); the CUDA
    path defines q0/eta := 0 when q0 == 0, so such a step is a pure prediction step."""
    d, r, T = 100, 6, 12
    Y, M, C0, x0 = make_problem(d, r, T, seed=4)
    M[6] = 0
    Y = Y * M
    X, Yrec, scal, st, _ = _engine_run(d, r, Y, M, C0, x0, impute_init(r), True)
    assert np.isfinite(X).all() and np.isfinite(st["C"]).all() and np.isfinite(st["V"]).all()
    assert np.array_equal(X[6], X[5])          # no observation: x_t = x_bar


def test_chunked_runs_carry_state():
    d, r, T = 700, 16, 48
    Y, M, C0, x0 = make_problem(d, r, T, seed=11)
    init = impute_init(r)
    one = _engine_run(d, r, Y, M, C0, x0, init, True)
    many = _engine_run(d, r, Y, M, C0, x0, init, True, chunks=[0, 1, 2, 17, 48])
    assert relerr(many[0], one[0]) < 1e-13
    assert relerr(many[3]["C"], one[3]["C"]) < 1e-13
    _compare(many, _oracle_run(Y, M, C0, x0, init, po.OracleConfig(robust=True)), TOL)


def test_run_to_run_determinism():
    d, r, T = 4000, 16, 20
    Y, M, C0, x0 = make_problem(d, r, T, seed=5)
    init = impute_init(r)
    a = _engine_run(d, r, Y, M, C0, x0, init, True)
    b = _engine_run(d, r, Y, M, C0, x0, init, True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[3]["C"], b[3]["C"])


def _workload_L_on_device(T, dtype, nan_encoded=False):
    """Workload L of bench.py (d = 1M, r = 16, rPSMF, 20 % missing) generated on the device by the bench generator."""
    import os
    import sys
    torch = _torch()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench_data as bd
    d, r = 1_000_000, 16
    Y, M, C0, x0 = bd.make_series(torch, torch.device("cuda", 0), d, 0, d, r, T, dtype, nan_encoded=nan_encoded)
    return d, r, Y, M, C0, x0, bd.init_state(r)


@pytest.mark.parametrize("dtype,T,tol", [("f64", 600, TOL), ("f32", 300, 1e-4)])
def test_full_size_workload_L_long_horizon(dtype, T, tol):
    """BASELINE.json's headline shape over HUNDREDS of steps (north_star: "over the full sequence"): lambda grows by d per
    step (to 6e8), rho and Q are multiplied by omega every step -- any drift of the pipelined statistics would show.
    The pipelined kernel, in several launches, against the C/OpenMP oracle (itself pinned against the numpy oracle in the
    CPU suite) at every step of x_t and at the end for C, P, V, rho, lambda; fp32 storage against the oracle on
    fp32-rounded inputs at 1e-4.  Size-independent properties: never-observed rows keep their C row bit-exactly."""
    from oracle import psmf_oracle_c as pc
    if not pc.available():
        pytest.skip("oracle/libpsmf_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    pc.use_all_cores()
    tdt = torch.float64 if dtype == "f64" else torch.float32
    d, r, Y, M, C0, x0, init = _workload_L_on_device(T, tdt)
    dead = torch.tensor([0, 31, 32, 4097, 500_000, d - 1], device="cuda")
    M[:, dead] = 0
    Y[:, dead] = 0
    C0 = C0.to(tdt)
    eng = FilterEngine(d, r, dtype=tdt, robust=True)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Xs = []
    bounds = [0, 1, 250, T]
    for a, b in zip(bounds[:-1], bounds[1:]):
        Xs.append(eng.run(Y[a:b], M[a:b], k0=1 + a, want_X=True)["X"])
        assert eng.status() == -1
    info = eng.launch_info()
    assert info["kernel"] == "tma" and info["resident"] is False
    X = torch.cat(Xs).cpu().numpy()
    st = eng.get_state()
    ref = pc.run(C0.double().cpu().numpy(), x0.numpy(), init["P"], init["V"], init["Q"], init["rho"], init["lam"],
                 Y.double().cpu().numpy(), M.cpu().numpy(), robust=True, cupdate_vt=True)
    assert ref["bad"] == -1
    per_step = np.max(np.abs(X - ref["X"]), axis=1) / np.max(np.abs(ref["X"]))
    assert per_step.max() < tol, (int(per_step.argmax()), float(per_step.max()))
    C = st["C"].double().cpu().numpy()
    assert relerr(C, ref["C"]) < tol
    assert relerr(st["P"].cpu().numpy(), ref["P"]) < tol and relerr(st["V"].cpu().numpy(), ref["V"]) < tol
    assert relerr(st["rho"].cpu().numpy(), ref["rho"]) < tol and relerr(st["lam"].cpu().numpy(), ref["lam"]) < 1e-12
    dd = dead.cpu().numpy()
    assert np.array_equal(C[dd], C0.double().cpu().numpy()[dd])
    eng.close()


def test_full_size_workload_L():
    """The headline shape on a short prefix with host-generated data: run-to-run bit-identity and both mask encodings."""
    from oracle import psmf_oracle_c as pc
    if not pc.available():
        pytest.skip("oracle/libpsmf_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    pc.use_all_cores()
    d, r, T = 1_000_000, 16, 6
    Y, M, C0, x0 = make_problem(d, r, T, seed=2026)
    dead = np.array([0, 31, 32, 4097, 500_000, d - 1])
    M[:, dead] = 0
    Y[:, dead] = 0.0
    init = impute_init(r)
    a = _engine_run(d, r, Y, M, C0, x0, init, True)
    assert a[4]["kernel"] == "tma" and a[4]["resident"] is False
    ref = pc.run(C0, x0, init["P"], init["V"], init["Q"], init["rho"], init["lam"], Y, M, robust=True, cupdate_vt=True)
    assert ref["bad"] == -1
    assert relerr(a[0], ref["X"]) < TOL
    assert relerr(a[3]["C"], ref["C"]) < TOL
    assert relerr(a[3]["P"], ref["P"]) < TOL and relerr(a[3]["V"], ref["V"]) < TOL
    assert relerr(a[3]["rho"], ref["rho"]) < TOL and relerr(a[3]["lam"], ref["lam"]) < TOL
    assert np.array_equal(a[3]["C"][dead], C0[dead])
    b = _engine_run(d, r, Y, M, C0, x0, init, True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[3]["C"], b[3]["C"])
    Yn = Y.copy()
    Yn[M == 0] = np.nan
    c = _engine_run(d, r, Yn, None, C0, x0, init, True, nan_mask=True)      # NaN-encoded mask: the same bits
    assert np.array_equal(a[0], c[0]) and np.array_equal(a[3]["C"], c[3]["C"])


@pytest.mark.parametrize("d,kernel", [(2_000_000, "tma"), (3_000_000, "direct")])
def test_very_large_shards(d, kernel):
    """Beyond the headline size on one GPU: at d = 2M the ring shrinks to 5 chunk slots; at d = 3M the residual
    buffer leaves no room for a ring and the engine must pick the direct-load kernel on its own."""
    from oracle import psmf_oracle_c as pc
    if not pc.available():
        pytest.skip("oracle/libpsmf_oracle.so not built")
    pc.use_all_cores()
    r, T = 16, 3
    Y, M, C0, x0 = make_problem(d, r, T, seed=3)
    init = impute_init(r)
    a = _engine_run(d, r, Y, M, C0, x0, init, True)
    assert a[4]["kernel"] == kernel
    ref = pc.run(C0, x0, init["P"], init["V"], init["Q"], init["rho"], init["lam"], Y, M, robust=True, cupdate_vt=True)
    assert relerr(a[0], ref["X"]) < TOL and relerr(a[3]["C"], ref["C"]) < TOL and relerr(a[3]["V"], ref["V"]) < TOL


def test_zero_initial_state_both_kernels():
    """x0 = 0 with random-walk dynamics (a Beijing-style init): a = xbar'V xbar = 0 at step 0, so w0 = 1/a = inf.
    Without missing rows the reference stays finite (Rbar = R + 0); both kernels must as well and agree with the
    oracle (the pipelined kernel builds s from q1 and q0 and must not form inf * 0)."""
    d, r, T = 3840, 16, 10
    Y, _, C0, _ = make_problem(d, r, T, seed=31, missing=0.0)
    x0 = np.zeros(r)
    init = impute_init(r)
    ref = _oracle_run(Y, None, C0, x0, init, po.OracleConfig(robust=True))
    assert np.isfinite(ref[1]).all()
    for kernel in (1, 2):
        res = _engine_run(d, r, Y, None, C0, x0, init, True, kernel=kernel)
        assert np.isfinite(res[0]).all() and np.isfinite(res[2]).all()
        _compare(res, ref, TOL)


def test_nearly_noise_free_data_kernels_agree():
    """The pipelined kernel rebuilds q1 = gamma - 2 xbar'h + xbar'A xbar from raw second moments; on a fit whose
    residual is far below the signal this cancels (relative accuracy of q1 ~ eps * gamma / q1).  Documented limit:
    q1 is clamped at 0, everything stays finite, and the two kernels still agree far better than the data noise."""
    d, r, T = 7680, 8, 30
    rng = np.random.RandomState(5)
    Ct = rng.randn(d, r)
    x = rng.randn(r)
    Y = np.zeros((T, d))
    for t in range(T):
        x = x + 0.1 * rng.randn(r)
        Y[t] = Ct @ x + 1e-7 * rng.randn(d)
    M = (rng.rand(T, d) >= 0.2).astype(np.uint8)
    Y = Y * M
    init = impute_init(r)
    x0 = x - 0.1 * rng.randn(r)
    a = _engine_run(d, r, Y, M, Ct, x0, init, True, kernel=1)
    b = _engine_run(d, r, Y, M, Ct, x0, init, True, kernel=2)
    assert a[4]["kernel"] == "direct" and b[4]["kernel"] == "tma"
    for res in (a, b):
        assert np.isfinite(res[0]).all() and np.isfinite(res[2]).all() and np.isfinite(res[3]["C"]).all()
        assert (res[2][:, 3] > 0).all() and (res[2][:, 4] > 0).all()          # omega, phi
    assert relerr(b[0], a[0]) < 1e-6 and relerr(b[3]["C"], a[3]["C"]) < 1e-6
    _compare(a, _oracle_run(Y, M, Ct, x0, init, po.OracleConfig(robust=True)), TOL)


def test_fp32_storage():
    torch = _torch()
    d, r, T = 600, 16, 40
    Y, M, C0, x0 = make_problem(d, r, T, seed=21)
    init = impute_init(r)
    res = _engine_run(d, r, Y, M, C0, x0, init, True, dtype=torch.float32)
    # the oracle sees the same fp32-rounded inputs
    ref = _oracle_run(Y.astype(np.float32).astype(np.float64), M, C0.astype(np.float32).astype(np.float64), x0, init,
                      po.OracleConfig(robust=True))
    _compare(res, ref, 1e-4)


def test_batched_series():
    torch = _torch()
    from rpsmf_b200 import FilterEngine
    S, d, r, T = 7, 96, 8, 30
    Y, M, C0, x0 = make_problem(d, r, T, seed=2, S=S)
    init = impute_init(r)
    eng = FilterEngine(d, r, n_series=S, robust=True)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    out = eng.run(torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda(), want_X=True, want_Yrec=True, want_scal=True)
    assert eng.status() == -1
    st = eng.get_state()
    for s in range(S):
        ost, oX, oYrec, oscal = _oracle_run(Y[s], M[s], C0[s], x0[s], init, po.OracleConfig(robust=True))
        assert relerr(out["X"][s].cpu().numpy(), oX) < TOL
        assert relerr(out["Yrec"][s].cpu().numpy(), oYrec) < TOL
        assert relerr(st["C"][s].cpu().numpy(), ost.C) < TOL
        assert relerr(st["P"][s].cpu().numpy(), ost.P) < TOL
    eng.close()


@pytest.mark.parametrize("tag,robust", [("psmf_full", False), ("rpsmf_full", True), ("rpsmf_scaled", True)])
def test_pypsmf_fixture_cos_dynamics(tag, robust):
    from rpsmf_b200 import _capi
    g = load_golden("pypsmf_cases")
    Y = g[tag + "_Y"]
    T, d = Y.shape
    C0 = g[tag + "_C0"]
    r = C0.shape[1]
    alpha = float(g[tag + "_alpha"]) if (tag + "_alpha") in g else 1.0
    beta = float(g[tag + "_beta"]) if (tag + "_beta") in g else 1.0
    init = dict(V=g[tag + "_V0"], P=g[tag + "_P0"], Q=g[tag + "_Q"], rho=float(g[tag + "_rho"]),
                lam=float(g[tag + "_lam0"]) if robust else 0.0, theta=g[tag + "_theta0"])
    X, Yrec, scal, st, _ = _engine_run(d, r, Y, None, C0, g[tag + "_mu0"], init, robust, dynamics=_capi.DYN_COS,
                                       alpha=alpha, beta=beta)
    assert relerr(Yrec, g[tag + "_ypred"]) < TOL
    assert relerr(st["C"], g[tag + "_C"]) < TOL
    assert relerr(st["x"], g[tag + "_mu"]) < TOL
    assert relerr(st["P"], g[tag + "_P"]) < TOL
    assert relerr(st["V"], g[tag + "_V"]) < TOL
    if robust:
        assert relerr(st["lam"], g[tag + "_lam_T"]) < TOL
        assert relerr(st["rho"], g[tag + "_rho_T"]) < TOL


@pytest.mark.parametrize("tag,robust", [("syn_psmf", False), ("syn_rpsmf", True)])
def test_simplified_mode_fixture(tag, robust):
    from rpsmf_b200 import _capi
    g = load_golden("pypsmf_cases")
    Y = g[tag + "_Y"]
    T, d = Y.shape
    C0 = g[tag + "_C0"]
    r = C0.shape[1]
    init = dict(V=g[tag + "_V0"], P=np.zeros((r, r)), Q=np.zeros((r, r)), rho=1.0, lam=1.8 if robust else 0.0,
                theta=g[tag + "_thetas"][0])
    X, Yrec, scal, st, _ = _engine_run(d, r, Y, None, C0, np.zeros(r), init, robust, dynamics=_capi.DYN_COS,
                                       simplified=True)
    assert relerr(st["C"], g[tag + "_Cs"][0]) < TOL
    assert relerr(st["x"], g[tag + "_mus"][0]) < TOL


def test_external_dynamics_stepwise():
    """PSMF_DYN_EXTERNAL: the host supplies x_bar and a dense F for every step (arbitrary callables)."""
    torch = _torch()
    from rpsmf_b200 import FilterEngine, _capi
    d, r, T = 150, 5, 12
    Y, M, C0, x0 = make_problem(d, r, T, seed=9)
    init = impute_init(r)
    rng = np.random.RandomState(0)
    A = np.eye(r) + 0.05 * rng.randn(r, r)
    eng = FilterEngine(d, r, robust=True, dynamics=_capi.DYN_EXTERNAL)
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    st = po.OracleState(C0.copy(), x0.copy(), init["P"].copy(), init["V"].copy(), init["Q"].copy(), init["rho"], init["lam"])
    cfg = po.OracleConfig(robust=True)
    Yd, Md = torch.as_tensor(Y).cuda(), torch.as_tensor(M).cuda()
    for t in range(T):
        xbar = np.tanh(A @ st.x)
        F = (1 - xbar ** 2)[:, None] * A
        st, out = po.step(st, cfg, Y[t], M[t].astype(float), xbar_F=(xbar, F))
        xg = eng.get_state(want_C=False)["x"].cpu().numpy()
        xbar_g = np.tanh(A @ xg)
        Fg = (1 - xbar_g ** 2)[:, None] * A
        res = eng.run(Yd[t:t + 1], Md[t:t + 1], k0=t + 1, xbar=xbar_g, F=Fg)
        assert relerr(res["X"][0].cpu().numpy(), st.x) < TOL
    gs = eng.get_state()
    assert relerr(gs["C"].cpu().numpy(), st.C) < TOL
    assert relerr(gs["P"].cpu().numpy(), st.P) < TOL
    eng.close()


@pytest.mark.parametrize("name", ["impute_pm25_30", "impute_pm10_head_20", "impute_sp500_head_30"])
@pytest.mark.parametrize("method", ["rPSMF", "PSMF"])
def test_impute_functions_against_reference_fixtures(name, method):
    """The drop-in flat functions reproduce what the unmodified reference returned (and, for PM25, published)."""
    from rpsmf_b200 import ProbabilisticSequentialMatrixFactorizer, robust_PSMF
    g = load_golden(name)
    c = impute_case(g)
    r = c["r"]
    d, n = c["Y"].shape
    X = c["X0"].copy()
    C = c["C0"].copy()
    pre = "rep0_%s_" % method
    Einit = float(g[pre + "Einit"])
    V, Q, R, P = 2 * np.eye(r), 0.1 * np.eye(r), 10 * np.eye(d), np.eye(r)
    if method == "rPSMF":
        ep, ef, rt, ib = robust_PSMF(c["Y"], C, X, d, n, r, c["M"], c["Mmiss"], V, Q, R, P, 1.8, 2, c["Iter"], c["YorigInt"], Einit)
    else:
        ep, ef, rt, ib = ProbabilisticSequentialMatrixFactorizer(c["Y"], C, X, d, n, r, c["M"], c["Mmiss"], 0, V, Q, R, P, 2,
                                                                 c["Iter"], c["YorigInt"], Einit)
    assert np.array_equal(C, c["C0"])                      # C is not mutated (rPSMF.py:111 rebinds)
    assert relerr(X, g[pre + "X_final"]) < TOL             # X is (rPSMF.py:104)
    assert relerr(ep, g[pre + "Epred"]) < TOL
    assert relerr(ef, g[pre + "Efull"]) < TOL
    assert abs(ib - float(g[pre + "inside"])) < 1e-12
    assert ep.shape == (1, c["Iter"] + 1) and rt.shape == (1, c["Iter"] + 1)
    if (pre + "published") in g:
        pub = g[pre + "published"]
        assert abs(ep[0, -1] - pub[0]) / pub[0] < 1e-9
        assert abs(ef[0, -1] - pub[1]) / pub[1] < 1e-9
        assert abs(ib - pub[2]) < 1e-12
