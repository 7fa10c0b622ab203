# -*- coding: utf-8 -*-
"""Host-side handle on the CUDA filter engine (thin wrapper over the C ABI).

PyTorch is used for device memory and streams only; every arithmetic step of
the filter runs in libpsmf_b200.so.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _capi


def _dev_tensor(a, dtype, device):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device).contiguous()


class FilterEngine:
    """One engine = one (batch of) series on one GPU.

    Parameters mirror ``psmf_config`` in include/psmf_b200.h.  ``grad_linear`` (linear dynamics only) makes
    ``run(want_grad=True)`` return the gradient of the summed incremental log-likelihood with respect to A and c
    (``grad_A`` (S, r, r), ``grad_c`` (S, r)) instead of ``grad``.  ``loglik`` makes the per-step scalar record 10 wide:
    ``run(want_loglik=True)`` returns ``nll`` (the incremental negative log-likelihood that the gradients differentiate) and
    ``logpred`` (the one-step predictive log-density log p(y_obs,k | y_<k)), each (S, T) float64 (include/psmf_b200.h
    PSMF_LOGLIK).

    ``n_series`` > 1 batches independent series in one launch.  A series runs on one CTA while it fits one (``ctas`` = 0);
    longer series, or ``ctas`` = c in 2..16, run on a thread-block cluster of c CTAs per series that sums its statistics
    through distributed shared memory.  That launch is not cooperative: clusters run in waves when there are more than the
    device holds at once.  ``launch_info()["ctas"]`` reports the CTAs per series.

    Smoothing: ``run(want_moments=True)`` (or ``moments_out``) returns the per-step moment record ``moments`` (S, T, NMOM(r))
    float64 (include/psmf_b200.h psmf_set_moments), and ``smooth(moments)`` runs the fixed-interval (RTS) smoother over it on
    the device.
    """

    def __init__(self, d, r, *, n_series=1, dtype=torch.float64, robust=True, simplified=False,
                 c_update_transpose=True, fixed_lambda=False, ll_student=False, dynamics=_capi.DYN_IDENTITY, alpha=1.0,
                 beta=1.0, device=None, d_global=None, world_size=1, rank=0, ctas=0, kernel=0, nan_mask=False,
                 exchange="nvlink", rho_vector=False, grad_linear=False, loglik=False):
        if not torch.cuda.is_available():
            raise RuntimeError("rpsmf_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if dtype not in (torch.float64, torch.float32):
            raise ValueError("dtype must be torch.float64 or torch.float32")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.d, self.r, self.S = int(d), int(r), int(n_series)
        self.dtype = dtype
        self.robust = bool(robust)
        flags = 0
        flags |= _capi.ROBUST if robust else 0
        flags |= _capi.SIMPLIFIED if simplified else 0
        flags |= _capi.CUPDATE_VT if c_update_transpose else 0
        flags |= _capi.FIXED_LAMBDA if fixed_lambda else 0
        flags |= _capi.LL_STUDENT if ll_student else 0
        flags |= _capi.NAN_MASK if nan_mask else 0
        flags |= _capi.RHO_VECTOR if rho_vector else 0
        flags |= _capi.GRAD_LINEAR if grad_linear else 0
        flags |= _capi.LOGLIK if loglik else 0
        self.loglik = bool(loglik)
        self.grad_linear = bool(grad_linear)
        self.rho_vector = bool(rho_vector)
        self.nan_mask = bool(nan_mask)
        if exchange not in ("nvlink", "external"):
            raise ValueError("exchange must be 'nvlink' (in-kernel mailboxes) or 'external' (caller-supplied collective)")
        self.exchange = exchange
        cfg = _capi.PsmfConfig(
            d=self.d, d_global=int(d_global or d), r=self.r, n_series=self.S,
            dtype=_capi.F64 if dtype == torch.float64 else _capi.F32, flags=flags, dynamics=int(dynamics),
            device=self.device.index, world_size=int(world_size), rank=int(rank), ctas=int(ctas), kernel=int(kernel),
            alpha=float(alpha), beta=float(beta), exchange=_capi.XCHG_EXTERNAL if exchange == "external" else _capi.XCHG_NVLINK,
            reserved=0)
        self._L = _capi.lib()
        self._h = C.c_void_p()
        rc = self._L.psmf_create(C.byref(self._h), C.byref(cfg))
        if rc != 0:
            msg = self._L.psmf_last_error(None)
            raise _capi.PsmfError(rc, msg.decode() if msg else "psmf_create failed")
        self.dynamics = int(dynamics)
        self._keep = []

    # -- lifecycle ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            torch.cuda.synchronize(self.device)
            self._L.psmf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ck(self, rc):
        _capi.check(self._h, rc)

    # -- state -------------------------------------------------------------------------------------
    def set_state(self, C_=None, V=None, P=None, x=None, Q=None, rho=None, lam=None, theta=None):
        S, d, r = self.S, self.d, self.r
        f64 = torch.float64

        def prep(a, shape, dt):
            if a is None:
                return None
            t = _dev_tensor(a, dt, self.device)
            if t.numel() != int(np.prod(shape)):
                if t.numel() * S == int(np.prod(shape)):       # broadcast one state over the batch
                    t = t.reshape((1,) + tuple(shape[1:])).expand(shape).contiguous()
                else:
                    raise ValueError("state tensor has %d elements, expected %s" % (t.numel(), shape))
            return t.reshape(shape)

        ts = [prep(C_, (S, d, r), self.dtype), prep(V, (S, r, r), f64), prep(P, (S, r, r), f64), prep(x, (S, r), f64),
              prep(Q, (S, r, r), f64), prep(rho, (S, d) if self.rho_vector else (S,), f64), prep(lam, (S,), f64),
              prep(theta, (S, r), f64)]
        ptrs = [C.c_void_p(t.data_ptr()) if t is not None else None for t in ts]
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_set_state(self._h, *ptrs, self._stream()))
        self._keep = ts   # keep sources alive until the async copies are ordered behind later work

    def get_state(self, want_C=True):
        S, d, r = self.S, self.d, self.r
        f64 = torch.float64
        dev = self.device
        out = dict(
            C=torch.empty((S, d, r), dtype=self.dtype, device=dev) if want_C else None,
            V=torch.empty((S, r, r), dtype=f64, device=dev), P=torch.empty((S, r, r), dtype=f64, device=dev),
            x=torch.empty((S, r), dtype=f64, device=dev), Q=torch.empty((S, r, r), dtype=f64, device=dev),
            rho=torch.empty((S, d) if self.rho_vector else (S,), dtype=f64, device=dev), lam=torch.empty((S,), dtype=f64, device=dev),
            theta=torch.empty((S, r), dtype=f64, device=dev))
        order = ("C", "V", "P", "x", "Q", "rho", "lam", "theta")
        ptrs = [C.c_void_p(out[k].data_ptr()) if out[k] is not None else None for k in order]
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_get_state(self._h, *ptrs, self._stream()))
        if self.S == 1:
            out = {k: (v[0] if v is not None else None) for k, v in out.items()}
        return out

    # -- the hot path ------------------------------------------------------------------------------
    def run(self, Y, M=None, k0=1, want_X=True, want_Yrec=False, want_scal=False, xbar=None, F=None,
            X_out=None, Yrec_out=None, scal_out=None, want_grad=False, Yorig=None, E=None, sig=2.0, want_loglik=False,
            want_moments=False, moments_out=None, _finish=False):
        """Filter ``T`` steps.  Y: device tensor (T, d) or (S, T, d) in the engine dtype (last dim may be
        padded: ld = stride of the time axis); M: uint8 tensor of the same shape or None.

        Fused evaluation (common.py:79-94): with ``E`` (uint8, 1 = evaluate here: the artificially removed entries)
        and ``Yorig`` (original values, same shape and strides as Y) the result holds ``eval`` = (S, 4) sums over this
        run: [sum (y_hat - y_orig)^2, entries inside y_hat -+ sig sqrt(U), entries of E, 0].

        ``want_loglik`` (an engine created with ``loglik=True``): ``nll`` and ``logpred``, (S, T) views of the 10-wide scalar
        record, which ``scal`` then is.

        ``want_moments`` / ``moments_out``: ``moments`` = (S, T, NMOM(r)) float64 record [x_bar | F | P_bar | x | P] of every
        step, the input of ``smooth``.  ``moments_out`` may be a view into a longer horizon (S, T_total, NMOM(r)) advanced by
        the steps already filtered; its series stride is kept.  The record is set for this launch only."""
        S, d, r = self.S, self.d, self.r
        if not isinstance(Y, torch.Tensor) or Y.device != self.device:
            raise ValueError("Y must be a tensor on %s" % self.device)
        if Y.dtype != self.dtype:
            raise ValueError("Y dtype %s does not match the engine dtype %s" % (Y.dtype, self.dtype))
        if Y.dim() == 2:
            Y = Y.unsqueeze(0)
        if Y.dim() != 3 or Y.shape[0] != S or Y.shape[2] < d or Y.stride(2) != 1:
            raise ValueError("Y must be (S, T, >=d) with unit stride along d")
        T = Y.shape[1]
        io = _capi.PsmfIO()
        io.Y, io.ldy, io.y_series_stride = Y.data_ptr(), Y.stride(1), Y.stride(0)
        if M is not None:
            if M.dtype != torch.uint8 or M.device != self.device:
                raise ValueError("M must be a uint8 tensor on %s" % self.device)
            if M.dim() == 2:
                M = M.unsqueeze(0)
            if M.shape[0] != S or M.shape[1] != T or M.shape[2] < d or M.stride(2) != 1:
                raise ValueError("M must be (S, T, >=d) with unit stride along d")
            io.M, io.ldm, io.m_series_stride = M.data_ptr(), M.stride(1), M.stride(0)
        res = {}
        if want_X or X_out is not None:
            X = X_out if X_out is not None else torch.empty((S, T, r), dtype=torch.float64, device=self.device)
            io.X_out = X.data_ptr()
            res["X"] = X
        if want_Yrec or Yrec_out is not None:
            Yr = Yrec_out if Yrec_out is not None else torch.empty((S, T, d), dtype=self.dtype, device=self.device)
            if Yr.dim() == 2:
                Yr = Yr.unsqueeze(0)
            io.Yrec_out, io.ldrec, io.rec_series_stride = Yr.data_ptr(), Yr.stride(1), Yr.stride(0)
            res["Yrec"] = Yr
        if want_loglik and not self.loglik:
            raise ValueError("want_loglik needs an engine created with loglik=True")
        if want_scal or want_loglik or scal_out is not None:
            nsc = _capi.NSCAL_LL if self.loglik else _capi.NSCAL
            sc = scal_out if scal_out is not None else torch.empty((S, T, nsc), dtype=torch.float64, device=self.device)
            if self.loglik and (sc.shape[-1] != nsc or not sc.is_contiguous()):
                raise ValueError("scal_out of a loglik engine must be a contiguous (S, T, %d) tensor" % nsc)
            io.scal_out = sc.data_ptr()
            res["scal"] = sc
            if want_loglik:
                res["nll"], res["logpred"] = sc[..., _capi.SCAL_NLL], sc[..., _capi.SCAL_LOGPRED]
        if want_grad:
            gr = torch.zeros((S, r * r + r if self.grad_linear else r), dtype=torch.float64, device=self.device)
            io.grad_out = gr.data_ptr()
            if self.grad_linear:                      # [G_A row-major | G_c] per series
                res["grad_A"], res["grad_c"] = gr[:, : r * r].view(S, r, r), gr[:, r * r:]
            else:
                res["grad"] = gr
        keep = [Y, M]
        if E is not None:
            if Yorig is None:
                raise ValueError("fused evaluation needs Yorig together with E")
            if Yorig.dim() == 2:
                Yorig = Yorig.unsqueeze(0)
            if E.dim() == 2:
                E = E.unsqueeze(0)
            if Yorig.dtype != self.dtype or Yorig.stride() != Y.stride() or Yorig.shape != Y.shape:
                raise ValueError("Yorig must have the dtype, shape and strides of Y")
            if E.dtype != torch.uint8 or E.shape[0] != S or E.shape[1] != T or E.shape[2] < d or E.stride(2) != 1:
                raise ValueError("E must be a uint8 tensor (S, T, >=d) with unit stride along d")
            ev = torch.zeros((S, _capi.NEVAL), dtype=torch.float64, device=self.device)
            io.Yorig, io.E, io.lde, io.e_series_stride, io.sig, io.eval_out = (Yorig.data_ptr(), E.data_ptr(), E.stride(1), E.stride(0),
                                                                              float(sig), ev.data_ptr())
            res["eval"] = ev
            keep += [Yorig, E]
        if self.dynamics == _capi.DYN_EXTERNAL:
            if xbar is None:
                raise ValueError("external dynamics: every run needs xbar (and F unless simplified)")
            xb = _dev_tensor(xbar, torch.float64, self.device).reshape(S, r)
            io.xbar_ext = xb.data_ptr()
            keep.append(xb)
            if F is not None:
                Ft = _dev_tensor(F, torch.float64, self.device).reshape(S, r, r)
                io.F_ext = Ft.data_ptr()
                keep.append(Ft)
        mom = None
        if want_moments or moments_out is not None:
            nm = _capi.NMOM(r)
            mom = moments_out if moments_out is not None else torch.empty((S, T, nm), dtype=torch.float64, device=self.device)
            if mom.dim() == 2:
                mom = mom.unsqueeze(0)
            if (mom.dtype != torch.float64 or mom.device != self.device or tuple(mom.shape) != (S, T, nm) or mom.stride(2) != 1
                    or mom.stride(1) != nm):
                raise ValueError("moments_out must be a float64 (S, T, %d) tensor on %s, contiguous per series" % (nm, self.device))
            res["moments"] = mom
            keep.append(mom)
        with torch.cuda.device(self.device):
            if mom is not None:
                self._ck(self._L.psmf_set_moments(self._h, C.c_void_p(mom.data_ptr()), mom.stride(0)))
            try:
                if _finish:
                    self._ck(self._L.psmf_run_finish(self._h, C.byref(io), int(k0), self._stream()))
                else:
                    self._ck(self._L.psmf_run(self._h, C.byref(io), T, int(k0), self._stream()))
            finally:
                if mom is not None:
                    self._L.psmf_set_moments(self._h, None, 0)
        self._keep_run = keep
        if S == 1:
            res = {k: v[0] for k, v in res.items()}
        return res

    def run_host(self, Y_host, M_host=None, window=256, k0=1, want_X=True):
        """Filter a long HOST-resident sequence: Y_host (T, d) pinned CPU tensor in the engine dtype, M_host
        (T, d) uint8.  Windows of ``window`` steps are copied host->device on a side stream while the
        previous window is being filtered (double buffering); returns X (T, r) on the host (pinned).
        Single-series engines only.  Each window is one launch, so ``status()`` afterwards describes the last window only."""
        if self.S != 1:
            raise ValueError("run_host supports single-series engines")
        T, d = Y_host.shape[0], self.d
        dev = self.device
        key = (int(window), int(Y_host.shape[1]), M_host is not None)
        if getattr(self, "_hb_key", None) != key:
            self._hb_key = key
            ld = Y_host.shape[1]
            self._hb = [torch.empty((window, ld), dtype=self.dtype, device=dev) for _ in range(2)]
            self._hm = [torch.empty((window, ld), dtype=torch.uint8, device=dev) for _ in range(2)] if M_host is not None else None
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._hx = torch.empty((2, window, self.r), dtype=torch.float64, device=dev)
        Xh = torch.empty((T, self.r), dtype=torch.float64).pin_memory() if want_X else None
        main = torch.cuda.current_stream(dev)
        cs = self._copy_stream
        cs.wait_stream(main)                        # staging buffers may still be read by an earlier run_host call
        nwin = (T + window - 1) // window
        copied = [None, None]
        done = [None, None]

        def issue_copy(w):
            a, b = w * window, min(T, (w + 1) * window)
            slot = w & 1
            if done[slot] is not None:
                cs.wait_event(done[slot])          # the run that last read this slot has finished
            with torch.cuda.stream(cs):
                self._hb[slot][: b - a].copy_(Y_host[a:b], non_blocking=True)
                if M_host is not None:
                    self._hm[slot][: b - a].copy_(M_host[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
            copied[slot] = ev

        issue_copy(0)
        for w in range(nwin):
            a, b = w * window, min(T, (w + 1) * window)
            slot = w & 1
            if w + 1 < nwin:
                issue_copy(w + 1)
            main.wait_event(copied[slot])
            out = self.run(self._hb[slot][: b - a], None if M_host is None else self._hm[slot][: b - a], k0=k0 + a,
                           want_X=False, X_out=self._hx[slot][: b - a].unsqueeze(0) if want_X else None)
            if want_X:
                Xh[a:b].copy_(self._hx[slot][: b - a], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(main)
            done[slot] = ev
        if want_X:
            done[(nwin - 1) & 1].synchronize()      # the returned host tensor is complete when the caller reads it
        return Xh

    # -- caller-driven statistics exchange (exchange="external") -----------------------------------------
    def stats_buffer(self):
        """The statistics vector of one step as a device tensor (a view of library memory, float64): after
        ``run`` it holds the sums over THIS GPU's rows; all-reduce it in place, then call ``run(..., _finish=True)``
        (or use ``run_split``)."""
        ptr, n = C.c_void_p(), C.c_int32()
        self._ck(self._L.psmf_stats_buffer(self._h, C.byref(ptr), C.byref(n)))
        if getattr(self, "_stats_view", None) is None:
            import ctypes
            # wrap the library's device buffer without copying: __cuda_array_interface__
            class _Arr:
                pass
            a = _Arr()
            a.__cuda_array_interface__ = dict(shape=(n.value,), typestr="<f8", data=(ptr.value, False), version=3)
            self._stats_view = torch.as_tensor(a, device=self.device)
        return self._stats_view

    def run_split(self, Y, M, k0, allreduce, **kw):
        """One filter step with the exchange done by the caller: pass + reduction of this GPU's rows, ``allreduce(buf)``
        (in place, sum over the GPUs that share the series; e.g. ``torch.distributed.all_reduce`` = ncclAllReduce on the
        current stream), then the r x r update and the rank-1 update of C.  Takes the keywords of ``run``.

        The pass writes the reconstruction, so ``Yrec_out`` / ``want_Yrec`` go to the first launch; X, the scalar record and
        the gradients come from the second.  External dynamics (``xbar``, ``F``) are read by both."""
        buf = self.stats_buffer()
        dyn = {k: kw[k] for k in ("xbar", "F") if k in kw}
        rec = kw.pop("Yrec_out", None)
        if kw.pop("want_Yrec", False) and rec is None:
            rec = torch.empty((self.S, Y.shape[-2], self.d), dtype=self.dtype, device=self.device)
        first = self.run(Y, M, k0=k0, want_X=False, Yrec_out=rec, **dyn)
        allreduce(buf)
        out = self.run(Y, M, k0=k0, _finish=True, **kw)
        if rec is not None:
            out["Yrec"] = first["Yrec"]
        return out

    # -- dynamics, forecast, evaluation ------------------------------------------------------------------
    def set_linear_dynamics(self, A, c=None):
        """PSMF_DYN_LINEAR: x_bar = A x + c, F = A."""
        At = _dev_tensor(A, torch.float64, self.device).reshape(self.r, self.r)
        ct = None if c is None else _dev_tensor(c, torch.float64, self.device).reshape(self.r)
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_set_linear_dynamics(self._h, C.c_void_p(At.data_ptr()), None if ct is None else C.c_void_p(ct.data_ptr()),
                                                      self._stream()))
        self._keep_lin = (At, ct)

    def predict(self, n_pred, k0, Xpred=None, want_Y=True):
        """Forecast n_pred steps from the current state (psmf.py:182-188): returns (Xpred (S, n_pred, r), Ypred
        (S, n_pred, d) or None).  ``Xpred`` replaces the device roll-out (external dynamics)."""
        S, d, r = self.S, self.d, self.r
        Xo = torch.empty((S, n_pred, r), dtype=torch.float64, device=self.device)
        Xi = None if Xpred is None else _dev_tensor(Xpred, torch.float64, self.device).reshape(S, n_pred, r)
        Yp = torch.empty((S, n_pred, d), dtype=self.dtype, device=self.device) if want_Y else None
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_predict(self._h, int(n_pred), int(k0), None if Xi is None else C.c_void_p(Xi.data_ptr()),
                                          C.c_void_p(Xo.data_ptr()), None if Yp is None else C.c_void_p(Yp.data_ptr()), d, n_pred * d,
                                          self._stream()))
        self._keep_pred = Xi
        if S == 1:
            return Xo[0], (None if Yp is None else Yp[0])
        return Xo, Yp

    def eval_full(self, X, Yorig, E):
        """Sum over the entries marked in E of (C X - Yorig)^2 with the engine's current C, and their number:
        (S, 2) device tensor (Efull of rPSMF.py:137-140 = sqrt(sum / count))."""
        S, r = self.S, self.r
        if Yorig.dim() == 2:
            Yorig = Yorig.unsqueeze(0)
        if E.dim() == 2:
            E = E.unsqueeze(0)
        X = X.reshape(S, -1, r).contiguous()
        n = X.shape[1]
        if Yorig.dtype != self.dtype or E.dtype != torch.uint8 or Yorig.shape[1] != n or E.shape[1] != n:
            raise ValueError("eval_full: Yorig (engine dtype) and E (uint8) must cover the n_steps of X")
        out = torch.empty((S, 2), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_eval_full(self._h, C.c_void_p(X.data_ptr()), n, C.c_void_p(Yorig.data_ptr()), Yorig.stride(1),
                                            Yorig.stride(0), C.c_void_p(E.data_ptr()), E.stride(1), E.stride(0),
                                            C.c_void_p(out.data_ptr()), self._stream()))
        self._keep_eval = (X, Yorig, E)
        return out

    def smooth(self, moments, want_P=False, check=True):
        """Fixed-interval (Rauch-Tung-Striebel) smoother over the moment record of ``run(want_moments=True)`` (S, T, NMOM(r)),
        one horizon of T steps, possibly written by several launches: returns Xs (S, T, r), and with ``want_P`` also Ps
        (S, T, r, r), float64 on the device.  Raises FloatingPointError on a non-finite result (a singular P_bar); with
        ``check=False`` the non-finite rows are returned as they are, for the caller to mask per series."""
        S, r = self.S, self.r
        nm = _capi.NMOM(r)
        mom = moments.unsqueeze(0) if moments.dim() == 2 else moments
        if (mom.dtype != torch.float64 or mom.device != self.device or mom.dim() != 3 or mom.shape[0] != S or mom.shape[2] != nm
                or mom.stride(2) != 1 or mom.stride(1) != nm):
            raise ValueError("moments must be a float64 (S, T, %d) tensor on %s, contiguous per series" % (nm, self.device))
        T = mom.shape[1]
        Xs = torch.empty((S, T, r), dtype=torch.float64, device=self.device)
        Ps = torch.empty((S, T, r, r), dtype=torch.float64, device=self.device) if want_P else None
        with torch.cuda.device(self.device):
            self._ck(self._L.psmf_smooth(self._h, C.c_void_p(mom.data_ptr()), mom.stride(0), T, C.c_void_p(Xs.data_ptr()),
                                         None if Ps is None else C.c_void_p(Ps.data_ptr()), self._stream()))
        if check and (not bool(torch.isfinite(Xs).all()) or (Ps is not None and not bool(torch.isfinite(Ps).all()))):
            raise FloatingPointError("smoother: non-finite smoothed moments (singular predicted covariance P_bar)")
        if S == 1:
            Xs, Ps = Xs[0], (None if Ps is None else Ps[0])
        return (Xs, Ps) if want_P else Xs

    def connect(self, dist):
        """Row sharding over several GPUs: exchange the mailbox blobs (CUDA IPC handle + plan record) through the
        process group `dist` (torch.distributed, any backend) and map every peer's mailbox.  The library derives
        the kernel choice from ALL ranks' records, so every rank runs the same kernel."""
        world = dist.get_world_size()
        buf = (C.c_ubyte * _capi.MAILBOX_BLOB_BYTES)()
        self._ck(self._L.psmf_mailbox_export(self._h, buf))
        mine = torch.tensor(list(bytes(buf)), dtype=torch.uint8)
        backend = dist.get_backend()
        if backend == "nccl":
            mine = mine.to(self.device)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        blob = b"".join(bytes(g.cpu().tolist()) for g in gathered)
        arr = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._ck(self._L.psmf_mailbox_connect(self._h, arr, world))
        dist.barrier()

    def status(self):
        """Synchronise and return the smallest step of the last launch, counted from 0 within that launch and taken over
        every series of the engine, at which a series produced a non-finite N/omega/phi/x or N == 0; -1 if there was none.
        Every launch starts the report afresh."""
        bad = C.c_int64(-1)
        self._ck(self._L.psmf_status(self._h, C.byref(bad)))
        return int(bad.value)

    def set_trace(self, steps):
        """Debug: record phase time stamps (ns, globaltimer) of CTA 0 for the first `steps` steps of each run."""
        self._trace = torch.zeros((steps * (16 + 320),), dtype=torch.int64, device=self.device) if steps else None
        self._ck(self._L.psmf_set_trace(self._h, C.c_void_p(self._trace.data_ptr()) if steps else None, int(steps)))
        return self._trace

    def launch_info(self):
        a, b, c, dd = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        self._ck(self._L.psmf_launch_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(dd)))
        k, ns, res = C.c_int32(), C.c_int32(), C.c_int32()
        self._ck(self._L.psmf_launch_info2(self._h, C.byref(k), C.byref(ns), C.byref(res)))
        return dict(ctas=a.value, threads=b.value, smem_bytes=c.value, launches=dd.value,
                    kernel={0: "none", 1: "direct", 2: "tma", 3: "batch"}[k.value], nslot=ns.value, resident=bool(res.value))


# -- handle-free device tools: ingest and the missing-segment generator ---------------------------------------
def _tool_ck(rc):
    if rc != 0:
        msg = _capi.lib().psmf_last_error(None)
        raise _capi.PsmfError(rc, msg.decode() if msg else "tool call failed")


def ingest(Ydn, dtype=torch.float64, keep_nan=False, want_mask=True, device=None):
    """(d, n) array with NaN = missing (the reference's data layout, rPSMF.py:160-164) -> time-major device tensors:
    Y (n, d) in ``dtype`` (NaN kept or zero-filled, rPSMF.py:200-202) and M (n, d) uint8 with 1 = observed
    (rPSMF.py:198).  The transpose and the NaN handling run on the device."""
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
    src = _dev_tensor(Ydn, torch.float64, dev)
    d, n = src.shape
    Y = torch.empty((n, d), dtype=dtype, device=dev)
    M = torch.empty((n, d), dtype=torch.uint8, device=dev) if want_mask else None
    with torch.cuda.device(dev):
        _tool_ck(_capi.lib().psmf_ingest(dev.index, C.c_void_p(src.data_ptr()), d, n, _capi.F64 if dtype == torch.float64 else _capi.F32,
                                         1 if keep_nan else 0, C.c_void_p(Y.data_ptr()), d, None if M is None else C.c_void_p(M.data_ptr()), d,
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return Y, M


def transpose_mask(Mdn, device=None):
    """(d, n) 0/1 array (any dtype; narrowed to one byte on the host) -> time-major (n, d) uint8 device tensor."""
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
    if isinstance(Mdn, torch.Tensor):
        src = (Mdn != 0).to(device=dev, dtype=torch.uint8).contiguous()
    else:
        src = torch.as_tensor(np.ascontiguousarray(np.asarray(Mdn) != 0).view(np.uint8)).to(dev)
    d, n = src.shape
    dst = torch.empty((n, d), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _tool_ck(_capi.lib().psmf_transpose_mask(dev.index, C.c_void_p(src.data_ptr()), d, n, C.c_void_p(dst.data_ptr()), d,
                                                 C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return dst


def missing_segments(Y_tm, E_tm, starts, seg=20):
    """One sweep of prepare_missing (common.py:66-75) on the device: Y_tm (n, d) NaN-encoded, E_tm (n, d) uint8, starts (d)
    integers from the caller's generator.  Returns the number of entries removed by this sweep."""
    dev = Y_tm.device
    n, d = Y_tm.shape
    st = torch.as_tensor(np.ascontiguousarray(starts, dtype=np.int64)).to(dev) if not isinstance(starts, torch.Tensor) else starts.to(dev, torch.int64)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _tool_ck(_capi.lib().psmf_missing_segments(dev.index, _capi.F64 if Y_tm.dtype == torch.float64 else _capi.F32,
                                                   C.c_void_p(Y_tm.data_ptr()), Y_tm.stride(0), C.c_void_p(E_tm.data_ptr()), E_tm.stride(0), d, n,
                                                   C.c_void_p(st.data_ptr()), int(seg), C.c_void_p(cnt.data_ptr()),
                                                   C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return int(cnt.item())


def count_nan(Y_tm):
    dev = Y_tm.device
    n, d = Y_tm.shape
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _tool_ck(_capi.lib().psmf_count_nan(dev.index, _capi.F64 if Y_tm.dtype == torch.float64 else _capi.F32, C.c_void_p(Y_tm.data_ptr()),
                                            Y_tm.stride(0), d, n, C.c_void_p(cnt.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return int(cnt.item())
