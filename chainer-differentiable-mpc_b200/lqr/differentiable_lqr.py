"""DiffLqr on B200 - the differentiable LQR layer of reference lqr/differentiable_lqr.py:21-142.

forward  = one fused Riccati + rollout launch that also stores K_t, Quu_t^-1, Qxu_t;
backward = the KKT adjoint (reference :78-142) re-using those factors instead of re-running
           the Riccati recursion, then lambda/d-lambda recursions and the outer products.
Gradient conventions follow the reference bit-for-bit by default (quirks Q1/Q2 of SURVEY.md);
pass strict_reference=False for the mathematically correct dC / df.

LqrNet / LqrNet_cost_dx (reference :145-248) are chainer.Links when Chainer is importable and plain objects with the
same call protocol otherwise; `backward_numpy` is their fused-reduction gradient path.
"""
import os
import sys

_here = os.path.dirname(os.path.abspath(__file__))
_pkg = os.path.dirname(_here)
for _p in (_pkg, _here):
    if _p not in sys.path:
        sys.path.append(_p)

import numpy as np  # noqa: E402

import _native  # noqa: E402
from _compat import HAVE_CHAINER, FunctionNodeBase, to_xp, wrap, as_f  # noqa: E402


class DiffLqr(FunctionNodeBase):
    """`DiffLqr(T, n_batch, n_state, n_ctrl).apply((x_init, C, c, F, f)) -> (x, u)`."""

    def __init__(self, T, n_batch, n_state, n_ctrl, device=0, dtype=np.float64, strict_reference=True,
                 pinned_outputs=False, context=None):
        super().__init__()
        self.T, self.n_batch, self.n_state, self.n_ctrl = int(T), int(n_batch), int(n_state), int(n_ctrl)
        self.n_sc = self.n_state + self.n_ctrl
        self.dtype = np.dtype(dtype)
        self.strict_reference = strict_reference
        self._ctx = context if context is not None else _native.default_context(device)
        self._d = None
        self._pinned = pinned_outputs
        self._host = {}
        self._have_f = False

    # ---- buffers -------------------------------------------------------------------------
    def _buffers(self):
        if self._d is None:
            T, B, n, m, s, dt, ctx = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype, self._ctx
            Tm = max(T - 1, 1)
            shapes = dict(x0=(B, n), C=(T, B, s, s), c=(T, B, s), F=(Tm, B, n, s), f=(Tm, B, n),
                          x=(T, B, n), u=(T, B, m), Ks=(T, B, m, n), ks=(T, B, m), fac=(ctx.lqr_fac_elems(T, B, n, m),),
                          gx=(T, B, n), gu=(T, B, m), dx0=(B, n), dC=(T, B, s, s), dc=(T, B, s),
                          dF=(Tm, B, n, s), df=(Tm, B, n))
            self._d = {k: ctx.empty(v, dt) for k, v in shapes.items()}
        return self._d

    def _host_buf(self, name, shape):
        """Fresh numpy array (reference semantics) or a re-used pinned buffer (bench e2e)."""
        if not self._pinned:
            return np.empty(shape, self.dtype)
        a = self._host.get(name)
        if a is None or a.shape != tuple(shape):
            a = self._ctx.pinned_empty(shape, self.dtype)
            self._host[name] = a
        return a

    # ---- numpy entry points (no Chainer needed) ---------------------------------------------
    def apply_numpy(self, x_init, C, c, large_f, f=None):
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        x_init, C, c = as_f(x_init, dt), as_f(C, dt), as_f(c, dt)
        assert list(x_init.shape) == [B, n]
        assert list(C.shape) == [T, B, s, s], "C dim mismatch"
        assert list(c.shape) == [T, B, s], "c dim mismatch"
        d = self._buffers()
        F = None
        if T > 1:
            F = as_f(large_f, dt)
            if F.shape[0] == T:
                F = F[:T - 1]
            assert list(F.shape) == [T - 1, B, n, s], "F dim mismatch"
        self._have_f = f is not None and to_xp(f) is not None
        if self._have_f and T > 1:
            f = as_f(f, dt)
            assert list(f.shape) == [T - 1, B, n], " f dim mismatch"
        ctx = self._ctx
        with _native.link_lock(ctx.device, "h2d"):      # one caller's upload burst at a time (see _native.link_lock)
            d["x0"].upload(x_init); d["C"].upload(C); d["c"].upload(c)
            if F is not None:
                d["F"].upload(F)
            if self._have_f and T > 1:
                d["f"].upload(f)
            ctx.sync()
        ctx.lqr_solve(dt, T, B, n, m, d["x0"], d["C"], d["c"], d["F"], T - 1, d["f"] if self._have_f else None,
                      d["x"], d["u"], d["Ks"], d["ks"], d["fac"],
                      _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
        x = d["x"].download(self._host_buf("x", (T, B, n)), sync=False)
        u = d["u"].download(self._host_buf("u", (T, B, m)))
        return x, u

    def apply_shared_numpy(self, x_init, C, c, large_f, f=None):
        """Shared-parameter entry: C [s,s], c [s], large_f [n,s] (and f [n] or None) are ONE block each, broadcast over
        [T, B] on the device (dmpc_expand_time_batch) instead of being repeated on the host and pushed through PCIe -
        what LqrNet / LqrNet_cost_dx do with util.expand_time_batch (reference differentiable_lqr.py:186-198, 237-248).
        Pair with backward_reduced_numpy, which returns the matching (T,B)-summed gradients."""
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        x_init = as_f(x_init, dt)
        C, c, Fm = as_f(C, dt), as_f(c, dt), as_f(large_f, dt)
        assert list(x_init.shape) == [B, n] and list(C.shape) == [s, s] and list(c.shape) == [s] and list(Fm.shape) == [n, s]
        d = self._buffers()
        ctx = self._ctx
        blk = ctx.to_device(np.concatenate((C.ravel(), c.ravel(), Fm.ravel(), np.zeros(n, dt) if f is None else as_f(f, dt).ravel())))
        d["x0"].upload(x_init)
        w = dt.itemsize
        ctx.expand_time_batch(dt, T, B, blk.ptr, d["C"], s * s)
        ctx.expand_time_batch(dt, T, B, blk.ptr + w * s * s, d["c"], s)
        if T > 1:
            ctx.expand_time_batch(dt, T - 1, B, blk.ptr + w * (s * s + s), d["F"], n * s)
            if f is not None:
                ctx.expand_time_batch(dt, T - 1, B, blk.ptr + w * (s * s + s + n * s), d["f"], n)
        self._have_f = f is not None
        ctx.lqr_solve(dt, T, B, n, m, d["x0"], d["C"], d["c"], d["F"], T - 1, d["f"] if self._have_f else None,
                      d["x"], d["u"], d["Ks"], d["ks"], d["fac"],
                      _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
        x = d["x"].download(self._host_buf("x", (T, B, n)), sync=False)
        u = d["u"].download(self._host_buf("u", (T, B, m)))
        return x, u

    def backward_numpy(self, grad_x, grad_u):
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        d = self._buffers()
        ctx = self._ctx
        d["gx"].upload(as_f(grad_x, dt)); d["gu"].upload(as_f(grad_u, dt))
        ctx.lqr_adjoint(dt, T, B, n, m, d["C"], d["c"], d["F"], d["x"], d["u"], d["gx"], d["gu"], d["Ks"],
                        d["fac"], d["dx0"], d["dC"], d["dc"], d["dF"], d["df"],
                        _native.ADJ_STRICT_REFERENCE if self.strict_reference else 0)
        Tm = max(T - 1, 1)
        ctx.sync()                                      # kernels done: take the download lane only for the copies
        with _native.link_lock(ctx.device, "d2h"):
            dx0 = d["dx0"].download(self._host_buf("dx0", (B, n)), sync=False)
            dC = d["dC"].download(self._host_buf("dC", (T, B, s, s)), sync=False)
            dc = d["dc"].download(self._host_buf("dc", (T, B, s)), sync=False)
            dF = d["dF"].download(self._host_buf("dF", (Tm, B, n, s)), sync=False)[:T - 1]
            df = d["df"].download(self._host_buf("df", (Tm, B, n)))[:T - 1]
        return dx0, dC, dc, dF, df

    def backward_reduced_numpy(self, grad_x, grad_u):
        """KKT adjoint with the (T,B)-sum fused in (dmpc_lqr_adjoint_reduced): returns
        (dx0 [B,n], sum dC [s,s], sum dc [s], sum dF [n,s], sum df [n]) - what a shared-parameter model
        (LqrNet, reference :186-198) receives after the backward of expand_time_batch - without materialising
        the [T,B,...] gradients."""
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        d = self._buffers()
        ctx = self._ctx
        rsz = ctx.reduced_grad_elems(n, m)
        if "partials" not in d:
            d["partials"] = ctx.empty((B, rsz), dt); d["sums"] = ctx.empty((rsz,), dt)
        d["gx"].upload(as_f(grad_x, dt)); d["gu"].upload(as_f(grad_u, dt))
        ctx.lqr_adjoint_reduced(dt, T, B, n, m, d["C"], d["c"], d["F"], d["x"], d["u"], d["gx"], d["gu"], d["Ks"],
                                d["fac"], d["dc"], d["partials"], d["dx0"], d["sums"],
                                _native.ADJ_STRICT_REFERENCE if self.strict_reference else 0)
        dx0 = d["dx0"].download(sync=False)
        sums = d["sums"].download()
        return (dx0,) + _native.Context.split_reduced(sums, n, m)

    # ---- Chainer FunctionNode protocol (reference :41-142) -----------------------------------
    def check_type_forward(self, in_types):
        pass

    def forward(self, inputs):
        x_init, C, c, large_f, f = inputs
        self.retain_inputs((0, 1, 2, 3))
        x, u = self.apply_numpy(x_init, C, c, large_f, f)
        self.retain_outputs((0, 1))
        return x, u

    def backward(self, target_input_indexes, grad_outputs):
        gx, gu = grad_outputs
        gx = np.zeros((self.T, self.n_batch, self.n_state), self.dtype) if to_xp(gx) is None else to_xp(gx)
        gu = np.zeros((self.T, self.n_batch, self.n_ctrl), self.dtype) if to_xp(gu) is None else to_xp(gu)
        return tuple(wrap(g) for g in self.backward_numpy(gx, gu))


class DiffLqrShared(FunctionNodeBase):
    """`DiffLqrShared(T, n_batch, n_state, n_ctrl).apply((x_init, C, c, F, f)) -> (x, u)` for a batch that shares its
    cost and dynamics matrices: C [T,s,s] and F [T-1 or T,n,s] are one block per time step; x_init [B,n] and
    f [T-1,B,n] (or None) are per element; c is per element [T,B,s] or shared [T,s] (chosen by c.ndim).  Same results
    as DiffLqr on the broadcast tensors; `backward` returns the gradients in the shapes of the inputs, dC, dF (and dc
    when c is [T,s]) summed over the batch (dmpc_lqr_solve_shared[_ex] / _adjoint_shared[_ex]: one Riccati sweep for
    the whole batch; with a shared c and f None the forward is that sweep plus the rollout)."""

    def __init__(self, T, n_batch, n_state, n_ctrl, device=0, dtype=np.float64, strict_reference=True, context=None):
        super().__init__()
        self.T, self.n_batch, self.n_state, self.n_ctrl = int(T), int(n_batch), int(n_state), int(n_ctrl)
        self.n_sc = self.n_state + self.n_ctrl
        self.dtype = np.dtype(dtype)
        self.strict_reference = strict_reference
        self._ctx = context if context is not None else _native.default_context(device)
        self._d = None
        self._F_T = None
        self._have_f = False
        self._shared_c = False

    def _buffers(self):
        if self._d is None:
            T, B, n, m, s, dt, ctx = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype, self._ctx
            Tm = max(T - 1, 1)
            shapes = dict(x0=(B, n), C=(T, s, s), F=(T, n, s), f=(Tm, B, n), x=(T, B, n), u=(T, B, m),
                          gx=(T, B, n), gu=(T, B, m), dx0=(B, n), dC=(T, s, s), dF=(T, n, s), df=(Tm, B, n))
            self._d = {k: ctx.empty(v, dt) for k, v in shapes.items()}
        d = self._d
        if self._shared_c and "ws_c" not in d:          # c [T,s]: dc [T,s] and the DMPC_SHARE_C workspace
            T, B, n, m, s, dt, ctx = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype, self._ctx
            d["c_s"], d["dc_s"] = ctx.empty((T, s), dt), ctx.empty((T, s), dt)
            d["ws_c"] = ctx.empty((ctx.lqr_shared_workspace_bytes(dt, T, B, n, m, _native.SHARE_C),), np.uint8)
        if not self._shared_c and "ws" not in d:        # c [T,B,s]
            T, B, n, m, s, dt, ctx = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype, self._ctx
            d["c"], d["dc"] = ctx.empty((T, B, s), dt), ctx.empty((T, B, s), dt)
            d["ws"] = ctx.empty((ctx.lqr_shared_workspace_bytes(dt, T, B, n, m),), np.uint8)
        return d

    def _mode(self):
        """(c buffer, dc buffer, workspace, share argument) of the form the last forward used."""
        d = self._d
        if self._shared_c:
            return d["c_s"], d["dc_s"], d["ws_c"], _native.SHARE_C
        return d["c"], d["dc"], d["ws"], None

    def apply_numpy(self, x_init, C, c, large_f, f=None):
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        x_init, C, c, F = as_f(x_init, dt), as_f(C, dt), as_f(c, dt), as_f(large_f, dt)
        assert list(x_init.shape) == [B, n]
        assert list(C.shape) == [T, s, s], "C dim mismatch"
        assert list(c.shape) in ([T, B, s], [T, s]), "c dim mismatch"
        assert F.shape[0] in (T - 1, T) and list(F.shape[1:]) == [n, s], "F dim mismatch"
        self._have_f = f is not None and to_xp(f) is not None and T > 1
        if self._have_f:
            f = as_f(f, dt)
            assert list(f.shape) == [T - 1, B, n], " f dim mismatch"
        self._F_T = F.shape[0]
        self._shared_c = c.ndim == 2
        d = self._buffers()
        c_buf, _, ws, share = self._mode()
        ctx = self._ctx
        d["x0"].upload(x_init); d["C"].upload(C); c_buf.upload(c)
        Fp = np.zeros((T, n, s), dt)                    # the device buffer has room for F_T = T rows
        Fp[:self._F_T] = F
        d["F"].upload(Fp)
        if self._have_f:
            d["f"].upload(f)
        ctx.lqr_solve_shared(dt, T, B, n, m, d["x0"], d["C"], c_buf, d["F"], self._F_T,
                             d["f"] if self._have_f else None, d["x"], d["u"], ws, share=share)
        x = d["x"].download(sync=False)
        u = d["u"].download()
        return x, u

    def backward_numpy(self, grad_x, grad_u):
        """-> (dx0 [B,n], dC [T,s,s], dc [T,B,s] (or [T,s], summed over the batch, when c was [T,s]), dF [F_T,n,s],
        df [T-1,B,n] or None)."""
        T, B, n, m, s, dt = self.T, self.n_batch, self.n_state, self.n_ctrl, self.n_sc, self.dtype
        d = self._buffers()
        c_buf, dc_buf, ws, share = self._mode()
        ctx = self._ctx
        gx = None if grad_x is None else d["gx"].upload(as_f(grad_x, dt))
        gu = None if grad_u is None else d["gu"].upload(as_f(grad_u, dt))
        ctx.lqr_adjoint_shared(dt, T, B, n, m, d["C"], c_buf, d["F"], self._F_T, d["x"], d["u"], gx, gu, ws,
                               d["dx0"], d["dC"], dc_buf, d["dF"], d["df"] if self._have_f else None,
                               _native.ADJ_STRICT_REFERENCE if self.strict_reference else 0, share=share)
        dx0 = d["dx0"].download(sync=False)
        dC = d["dC"].download(sync=False)
        dc = dc_buf.download(sync=False)
        df = d["df"].download(sync=False)[:T - 1] if self._have_f else None
        dF = d["dF"].download()[:self._F_T]
        return dx0, dC, dc, dF, df

    # ---- Chainer FunctionNode protocol -------------------------------------------------------
    def check_type_forward(self, in_types):
        pass

    def forward(self, inputs):
        x_init, C, c, large_f, f = inputs
        self.retain_inputs((0, 1, 2, 3))
        x, u = self.apply_numpy(x_init, C, c, large_f, f)
        self.retain_outputs((0, 1))
        return x, u

    def backward(self, target_input_indexes, grad_outputs):
        gx, gu = grad_outputs
        return tuple(None if g is None else wrap(g) for g in self.backward_numpy(to_xp(gx), to_xp(gu)))


from _compat import NetLinkBase, Parameter  # noqa: E402
from util import expand_batch, expand_time_batch  # noqa: E402


def _cat_ab(A, B):
    if HAVE_CHAINER:
        from chainer import functions as F
        return F.concat((A, B), axis=1)
    return np.concatenate((A.array, B.array), axis=1)


def _shared_fits(dtype, T, B, n, m, share=None):
    """False when the shared path's chunk kernels cannot hold the shape (dmpc_lqr_shared_workspace_bytes[_ex] reports
    DMPC_ERR_UNSUPPORTED); the per-element path (DiffLqr) runs every n <= 128, m <= 32."""
    try:
        _native.default_context().lqr_shared_workspace_bytes(dtype, T, B, n, m, share)
    except _native.DiffMpcError:
        return False
    return True


def _batch_invariant(C):
    """True when C [T,B,...] is a plain array whose entries do not vary along the batch axis: a stride-0 broadcast, or
    (checked second) a copy of C[:, :1]."""
    if not isinstance(C, np.ndarray) or C.ndim < 2 or C.shape[1] < 1:
        return False
    return C.strides[1] == 0 or np.array_equal(C, np.broadcast_to(C[:, :1], C.shape))


class LqrNet(NetLinkBase):
    """Learn A, B through the LQR layer (reference :145-198; same seeding, :167-171).  C and c come in as the reference
    takes them ([T,B,s,s], [T,B,s]).  When C is a plain array that does not vary over the batch (the LQRnet notebook's
    C = I), the layer is DiffLqrShared on C[:, 0] and the per-element c: one Riccati sweep for the batch, and
    `backward_numpy` sums dF over t on the host.  Otherwise (C varies per element, or is a Chainer Variable whose
    per-element dC the caller may read) it is DiffLqr, and `backward_numpy` is its fused path: the (T,B)-sum of dF inside
    the adjoint kernel -> A.grad, B.grad without the [T-1,B,n,s] tensor."""

    def __init__(self, T, n_batch, n_state, n_ctrl, seed):
        super().__init__()
        self.T, self.n_batch, self.n_state, self.n_ctrl = T, n_batch, n_state, n_ctrl
        self.n_sc = n_state + n_ctrl
        with self.init_scope():
            np.random.seed(seed)
            A = np.eye(n_state).astype("float") + 0.2 * np.random.randn(n_state, n_state).astype("float")
            self.A = Parameter(A)
            self.B = Parameter(np.random.randn(n_state, n_ctrl).astype("float"))
        self.lqr_layer = DiffLqr(T, n_batch, n_state, n_ctrl)
        self.lqr_shared = DiffLqrShared(T, n_batch, n_state, n_ctrl)
        self._used_shared = False

    def forward(self, inputs):
        x_init, C, c, f = inputs
        self._used_shared = _batch_invariant(C) and _shared_fits(np.float64, self.T, self.n_batch, self.n_state,
                                                                 self.n_ctrl)
        if self._used_shared:
            large_f = expand_batch(_cat_ab(self.A, self.B), self.T - 1)             # [T-1, n, s]
            return self.lqr_shared.apply((x_init, np.ascontiguousarray(C[:, 0]), c, large_f, f))
        large_f = expand_time_batch(_cat_ab(self.A, self.B), self.T - 1, self.n_batch)
        return self.lqr_layer.apply((x_init, C, c, large_f, f))

    def backward_numpy(self, grad_x, grad_u):
        n = self.n_state
        if self._used_shared:
            gF = self.lqr_shared.backward_numpy(grad_x, grad_u)[3].sum(0)           # sum over t of dF [T-1, n, s]
        else:
            gF = self.lqr_layer.backward_reduced_numpy(grad_x, grad_u)[3]           # (dx0, sum dC, sum dc, sum dF, sum df)
        self.A.grad, self.B.grad = gF[:, :n].copy(), gF[:, n:].copy()
        return self.A.grad, self.B.grad


class LqrNet_cost_dx(NetLinkBase):
    """Learn A, B, C, c (reference :201-248; C = I + 0.2 randn is NOT symmetric, Q10).  The layer is DiffLqrShared with
    C [T,s,s], c [T,s] and [A B] [T-1,n,s] broadcast over time only (util.expand_batch, so Chainer sums their gradients
    over t); x_init and f stay per element.  With f None the forward is one Riccati sweep plus the rollout.
    `backward_numpy` sums dC, dc and dF over t on the host."""

    def __init__(self, T, n_batch, n_state, n_ctrl, seed):
        super().__init__()
        self.T, self.n_batch, self.n_state, self.n_ctrl = T, n_batch, n_state, n_ctrl
        self.n_sc = n_state + n_ctrl
        with self.init_scope():
            np.random.seed(seed)
            self.A = Parameter(np.eye(n_state).astype("float") + 0.2 * np.random.randn(n_state, n_state).astype("float"))
            self.B = Parameter(np.random.randn(n_state, n_ctrl).astype("float"))
            self.C = Parameter(np.eye(self.n_sc).astype("float") + 0.2 * np.random.randn(self.n_sc, self.n_sc).astype("float"))
            self.c = Parameter(np.random.randn(self.n_sc).astype("float"))
        # shapes beyond the shared path's chunk kernels: host broadcast over [T, B], DiffLqr and its fused reduction
        self._shared = _shared_fits(np.float64, T, n_batch, n_state, n_ctrl, _native.SHARE_C)
        self.lqr_layer = (DiffLqrShared if self._shared else DiffLqr)(T, n_batch, n_state, n_ctrl)

    def forward(self, inputs):
        x_init, f = inputs
        if not self._shared:
            large_f = expand_time_batch(_cat_ab(self.A, self.B), self.T - 1, self.n_batch)
            C = expand_time_batch(self.C, self.T, self.n_batch)
            c = expand_time_batch(self.c, self.T, self.n_batch)
            return self.lqr_layer.apply((x_init, C, c, large_f, f))
        large_f = expand_batch(_cat_ab(self.A, self.B), self.T - 1)
        C = expand_batch(self.C, self.T)
        c = expand_batch(self.c, self.T)
        return self.lqr_layer.apply((x_init, C, c, large_f, f))

    def backward_numpy(self, grad_x, grad_u):
        n = self.n_state
        if not self._shared:
            g = self.lqr_layer.backward_reduced_numpy(grad_x, grad_u)       # (dx0, sum dC, sum dc, sum dF, sum df)
            self.C.grad, self.c.grad = g[1].copy(), g[2].copy()
            self.A.grad, self.B.grad = g[3][:, :n].copy(), g[3][:, n:].copy()
            return self.A.grad, self.B.grad, self.C.grad, self.c.grad
        g = self.lqr_layer.backward_numpy(grad_x, grad_u)                   # (dx0, dC [T,s,s], dc [T,s], dF, df)
        self.C.grad, self.c.grad = g[1].sum(0), g[2].sum(0)
        gF = g[3].sum(0)
        self.A.grad, self.B.grad = gF[:, :n].copy(), gF[:, n:].copy()
        return self.A.grad, self.B.grad, self.C.grad, self.c.grad
