"""ctypes binding of libdiffmpc_b200.so (C ABI: include/diffmpc_b200.h).

This is the only bridge between the Python facade modules (lqr/, mpc/) and the
sm_100a kernels.  There is NO CPU fallback: importing works without a GPU (so
the symbol table can be checked), but creating a context raises.
"""
import ctypes
import os

import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DIFFMPC_LIB points at another build of the SAME library (A/B runs of kernel variants under profiles/tools); the
# product default is the in-tree libdiffmpc_b200.so next to this file.
LIB_PATH = os.environ.get("DIFFMPC_LIB") or os.path.join(_HERE, "libdiffmpc_b200.so")

F64, F32 = 0, 1
LQR_FACTOR, LQR_ROLLOUT, LQR_SAVE_FAC = 1, 2, 4
ADJ_STRICT_REFERENCE = 1
ADJ_STAGE_DTAU_ONLY, ADJ_STAGE_OUT_ONLY = 2, 4
SHARE_C = 1
COUPLING_ELEMENT, COUPLING_BATCH = 0, 1
DYN_LINEAR, DYN_PENDULUM = 0, 1
FLAG_QP_NOT_CONVERGED, FLAG_NONFINITE, FLAG_LS_CAPPED, FLAG_BAD_BOUNDS = 1, 2, 4, 8

_vp = ctypes.c_void_p
_i = ctypes.c_int
_sz = ctypes.c_size_t
_d = ctypes.c_double

# name -> (restype, argtypes); must list every symbol declared in include/diffmpc_b200.h
SIGNATURES = {
    "dmpc_version": (_i, []),
    "dmpc_status_string": (ctypes.c_char_p, [_i]),
    "dmpc_create": (_i, [_i, ctypes.POINTER(_vp)]),
    "dmpc_destroy": (_i, [_vp]),
    "dmpc_last_error": (ctypes.c_char_p, [_vp]),
    "dmpc_device_count": (_i, []),
    "dmpc_malloc": (_i, [_vp, _sz, ctypes.POINTER(_vp)]),
    "dmpc_free": (_i, [_vp, _vp]),
    "dmpc_host_alloc": (_i, [_vp, _sz, ctypes.POINTER(_vp)]),
    "dmpc_host_free": (_i, [_vp, _vp]),
    "dmpc_memcpy_h2d": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "dmpc_memcpy_d2h": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "dmpc_memset": (_i, [_vp, _vp, _i, _sz, _vp]),
    "dmpc_sync": (_i, [_vp, _vp]),
    "dmpc_launch_count": (ctypes.c_longlong, [_vp]),
    "dmpc_lqr_fac_elems": (_sz, [_i, _i, _i, _i]),
    "dmpc_lqr_solve": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "dmpc_lqr_adjoint": (_i, [_vp, _i, _i, _i, _i, _i] + [_vp] * 14 + [_i, _vp]),
    "dmpc_pnqp": (_i, [_vp, _i, _i, _i] + [_vp] * 5 + [_i, _i] + [_vp] * 7),
    "dmpc_mpc_step_forward": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i,
                                   _vp, _vp, ctypes.POINTER(_d), _d, _i, _i, _i] + [_vp] * 14),
    "dmpc_mpc_step_backward": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i] + [_vp] * 15 + [_vp]),
    "dmpc_lqr_active_solve": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dmpc_get_traj": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, ctypes.POINTER(_d), _vp, _vp, _vp, _vp]),
    "dmpc_expand_time_batch": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "dmpc_warmstart_take": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "dmpc_warmstart_put": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "dmpc_reduced_grad_elems": (_sz, [_i, _i]),
    "dmpc_lqr_adjoint_reduced": (_i, [_vp, _i, _i, _i, _i, _i] + [_vp] * 13 + [_i, _vp]),
    "dmpc_mpc_step_backward_reduced": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i] + [_vp] * 13 + [_vp]),
    "dmpc_lqr_shared_workspace_bytes": (_i, [_i, _i, _i, _i, _i, ctypes.POINTER(_sz)]),
    "dmpc_lqr_solve_shared": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmpc_lqr_adjoint_shared": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz]
                                + [_vp] * 5 + [_i, _vp]),
    "dmpc_lqr_shared_workspace_bytes_ex": (_i, [_i, _i, _i, _i, _i, _i, ctypes.POINTER(_sz)]),
    "dmpc_lqr_solve_shared_ex": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _i,
                                      _vp]),
    "dmpc_lqr_adjoint_shared_ex": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz]
                                   + [_vp] * 5 + [_i, _i, _vp]),
    "dmpc_boxddp_workspace_bytes": (_i, [_i, _i, _i, _i, _i, ctypes.POINTER(_sz)]),
    "dmpc_boxddp_solve": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, ctypes.POINTER(_d), _vp,
                               _vp, _vp, _sz] + [_vp] * 7 + [ctypes.POINTER(_i)] * 3 + [_vp]),
}


class BoxDdpOpts(ctypes.Structure):
    """dmpc_boxddp_opts of include/diffmpc_b200.h."""
    _fields_ = [("eps", _d), ("best_cost_eps", _d), ("ls_decay", _d), ("not_improved_lim", _i), ("max_iter", _i),
                ("max_ls_trials", _i), ("coupling", _i), ("poll_every", _i)]


BOXDDP_MAX_ITER, BOXDDP_CONVERGED, BOXDDP_NOT_IMPROVED = 0, 1, 2

_lib = None


class DiffMpcError(RuntimeError):
    pass


def load_library():
    """dlopen the in-tree shared library and type every entry point.  Raises if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DiffMpcError(
            "libdiffmpc_b200.so not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C chainer-differentiable-mpc_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def dtype_code(dt):
    dt = np.dtype(dt)
    if dt == np.float64:
        return F64
    if dt == np.float32:
        return F32
    raise DiffMpcError("unsupported dtype %s (float64 / float32 only)" % dt)


# ---- host<->device link arbitration ---------------------------------------------------------------------
# A forward call is upload-heavy and a backward call download-heavy.  When several host threads feed one GPU
# (one Context each), letting each direction of the PCIe link serve ONE caller's burst at a time makes the
# callers fall into anti-phase (A downloads while B uploads) and keeps both directions busy; interleaving
# same-direction bursts would only stretch both.  One lock per (device, direction), process-wide.
_LINK_LOCKS = {}
_LINK_LOCKS_GUARD = threading.Lock()


def link_lock(device, direction):
    """`with link_lock(dev, "h2d"):` around a burst of uploads (or "d2h" downloads) including its stream sync."""
    key = (int(device), direction)
    with _LINK_LOCKS_GUARD:
        lk = _LINK_LOCKS.get(key)
        if lk is None:
            lk = _LINK_LOCKS[key] = threading.Lock()
    return lk


class DeviceArray:
    """A typed, shaped cudaMalloc'ed buffer owned by a Context."""

    def __init__(self, ctx, shape, dtype):
        self.ctx = ctx
        self.shape = tuple(int(v) for v in shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        self.ptr = ctx._alloc(self.nbytes)
        self._owned = True

    def upload(self, arr, stream=None):
        arr = np.ascontiguousarray(arr, dtype=self.dtype)
        assert arr.shape == self.shape, (arr.shape, self.shape)
        self.ctx._check(self.ctx.lib.dmpc_memcpy_h2d(self.ctx.h, self.ptr, arr.ctypes.data, self.nbytes, stream))
        # pageable memcpyAsync returns after staging, so `arr` may be released
        return self

    def download(self, out=None, stream=None, sync=True):
        if out is None:
            out = np.empty(self.shape, dtype=self.dtype)
        assert out.flags["C_CONTIGUOUS"] and out.nbytes == self.nbytes
        self.ctx._check(self.ctx.lib.dmpc_memcpy_d2h(self.ctx.h, out.ctypes.data, self.ptr, self.nbytes, stream))
        if sync:
            self.ctx.sync(stream)
        return out

    def zero(self, stream=None):
        self.ctx._check(self.ctx.lib.dmpc_memset(self.ctx.h, self.ptr, 0, self.nbytes, stream))
        return self

    def free(self):
        if self._owned and self.ptr and self.ctx.h:
            self.ctx._release(self.ptr, self.nbytes)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PackedBuffers:
    """Several typed device arrays carved from ONE allocation, so that a latency-bound call (a batch-64 MPC step
    moves a few hundred KB in ~20 tensors) needs one host->device and one device->host copy instead of one per
    tensor.  `views[name]` are non-owning DeviceArrays; `upload(dict)` stages the host arrays contiguously in a PINNED
    host buffer and issues one copy; `download()` returns copies of one device->host transfer.
    `acquire(ctx, specs)` / `release()` keep one instance per layout in the context: a step that is called again and
    again (BoxDDP's host loop, the latency benchmark) pays for the allocation and the page-locking once."""

    ALIGN = 256

    def __init__(self, ctx, specs):
        self.ctx = ctx
        self.layout = {}
        o = 0
        for name, shape, dtype in specs:
            dt = np.dtype(dtype)
            shape = tuple(int(v) for v in shape)
            nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
            self.layout[name] = (o, shape, dt, nbytes)
            o = (o + nbytes + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.total = max(o, self.ALIGN)
        self.base = DeviceArray(ctx, (self.total,), np.uint8)
        self.host = ctx.pinned_empty((self.total,), np.uint8)        # page-locked staging: copies run at PCIe speed
        self.views = {}
        self.hviews = {}                                             # typed host views of the staging buffer, built once
        self._key = None
        for name, (off, shape, dt, nbytes) in self.layout.items():
            v = DeviceArray.__new__(DeviceArray)
            v.ctx, v.shape, v.dtype, v.nbytes, v.ptr, v._owned, v._base = ctx, shape, dt, nbytes, self.base.ptr + off, False, self.base
            self.views[name] = v
            self.hviews[name] = self.host[off:off + nbytes].view(dt).reshape(shape)

    @classmethod
    def acquire(cls, ctx, specs, key=None):
        """`specs` = [(name, shape, dtype)] or a callable returning it (only evaluated on a cache miss); `key` = a cheap
        hashable that identifies the layout (callers on a latency path pass one instead of having it derived per call)."""
        if key is None:
            if callable(specs):
                specs = specs()
            key = tuple((n, tuple(int(v) for v in sh), np.dtype(dt).str) for n, sh, dt in specs)
        cache = ctx.__dict__.setdefault("_packed_cache", {})
        lst = cache.get(key)
        if lst:
            return lst.pop()
        pb = cls(ctx, specs() if callable(specs) else specs)
        pb._key = key
        return pb

    def release(self):
        if self._key is None:
            return self.free()
        self.ctx.__dict__.setdefault("_packed_cache", {}).setdefault(self._key, []).append(self)

    def upload(self, arrays, stream=None):
        hv = self.hviews
        for name, arr in arrays.items():
            h = hv[name]
            assert arr.shape == h.shape, (name, arr.shape, h.shape)
            h[...] = arr
        self.ctx._check(self.ctx.lib.dmpc_memcpy_h2d(self.ctx.h, self.base.ptr, self._host_ptr(), self.total, stream))
        return self.views

    def _host_ptr(self):
        p = self.__dict__.get("_hp")
        if p is None:
            p = self.__dict__["_hp"] = self.host.ctypes.data
        return p

    def download(self, stream=None):
        self.ctx._check(self.ctx.lib.dmpc_memcpy_d2h(self.ctx.h, self._host_ptr(), self.base.ptr, self.total, stream))
        self.ctx.sync(stream)
        return {name: h.copy() for name, h in self.hviews.items()}

    def free(self):
        self.base.free()


class WarmStartCache:
    """The warm-start cache of the reference's training loop (env_dx/il_exp.py:215-257: `train_warmstart[n_samples, T, m]`,
    read with the minibatch's sample ids, written back with the solver's controls, zeroed every `restart_warmstart_every`
    epochs) kept in HBM: `take(idxs)` returns the device tensor u_init[T, B, m] that BoxDDP accepts as is, `put(idxs, u)`
    stores the device tensor BoxDDP leaves in `solver.u_device` - no host round trip of the controls."""

    def __init__(self, ctx, n_samples, T, m, dtype=np.float64):
        self.ctx, self.n_samples, self.T, self.m, self.dtype = ctx, int(n_samples), int(T), int(m), np.dtype(dtype)
        self.cache = ctx.zeros((self.n_samples, self.T, self.m), self.dtype)

    def reset(self):
        self.cache.zero()

    def _idx(self, idxs):
        return self.ctx.to_device(np.ascontiguousarray(idxs, dtype=np.int32))

    def take(self, idxs):
        B = len(idxs)
        u = self.ctx.empty((self.T, B, self.m), self.dtype)
        self.ctx.warmstart_take(self.dtype, self.T, B, self.m, self.n_samples, self.cache, self._idx(idxs), u)
        return u

    def put(self, idxs, u):
        B = len(idxs)
        if not isinstance(u, DeviceArray):
            u = self.ctx.to_device(np.ascontiguousarray(u, dtype=self.dtype))
        assert tuple(u.shape) == (self.T, B, self.m) and u.dtype == self.dtype
        self.ctx.warmstart_put(self.dtype, self.T, B, self.m, self.n_samples, self.cache, self._idx(idxs), u)

    def download(self):
        return self.cache.download()


PACK_LIMIT_BYTES = 8 << 20      # above this the extra host-side staging copy costs more than the saved API calls


def _p(x):
    if x is None:
        return None
    if isinstance(x, DeviceArray):
        return x.ptr
    return int(x)       # raw device pointer (e.g. torch.Tensor.data_ptr())


class Context:
    """One handle per device (cudaStream + launch counter)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.h = None
        h = _vp()
        rc = self.lib.dmpc_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise DiffMpcError("dmpc_create(device=%d) failed: %s" % (device, self.lib.dmpc_status_string(rc).decode()))
        self.h = h
        self.device = int(device)
        self._pinned = []        # page-locked host allocations handed out by pinned_empty()
        self._pool = {}          # nbytes -> [device pointers]; avoids cudaMalloc/cudaFree per call
        self._pool_bytes = 0
        self.pool_limit = 8 << 30

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.dmpc_status_string(rc).decode()
            det = self.lib.dmpc_last_error(self.h).decode() if self.h else ""
            if rc in (1, 2, 3):
                raise AssertionError("%s: %s" % (msg, det))     # the reference raises AssertionError here
            raise DiffMpcError("%s: %s" % (msg, det))

    def _alloc(self, nbytes):
        lst = self._pool.get(nbytes)
        if lst:
            self._pool_bytes -= nbytes
            return lst.pop()
        p = _vp()
        rc = self.lib.dmpc_malloc(self.h, nbytes, ctypes.byref(p))
        if rc != 0 and self._pool:
            self.trim()
            rc = self.lib.dmpc_malloc(self.h, nbytes, ctypes.byref(p))
        self._check(rc)
        return p.value

    def _release(self, ptr, nbytes):
        if self._pool_bytes + nbytes > self.pool_limit:
            self.lib.dmpc_free(self.h, ptr)
            return
        self._pool.setdefault(nbytes, []).append(ptr)
        self._pool_bytes += nbytes

    def trim(self):
        """Return every cached buffer to the driver."""
        for lst in self._pool.values():
            for ptr in lst:
                self.lib.dmpc_free(self.h, ptr)
        self._pool.clear()
        self._pool_bytes = 0

    def close(self):
        if self.h:
            self.trim()
            for p in self._pinned:
                self.lib.dmpc_host_free(self.h, p)
            self._pinned = []
            self.lib.dmpc_destroy(self.h)
            self.h = None

    def sync(self, stream=None):
        self._check(self.lib.dmpc_sync(self.h, stream))

    def pinned_empty(self, shape, dtype=np.float64):
        """numpy array backed by page-locked host memory (dmpc_host_alloc): copies to / from it run at PCIe speed and
        truly asynchronously.  The memory lives until the context is closed."""
        dt = np.dtype(dtype)
        shape = tuple(int(v) for v in shape)
        nbytes = max(int(np.prod(shape, dtype=np.int64)) * dt.itemsize, 1)
        p = _vp()
        self._check(self.lib.dmpc_host_alloc(self.h, nbytes, ctypes.byref(p)))
        self._pinned.append(p)
        buf = (ctypes.c_ubyte * nbytes).from_address(p.value)
        return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)

    @property
    def launches(self):
        return int(self.lib.dmpc_launch_count(self.h))

    def empty(self, shape, dtype=np.float64):
        return DeviceArray(self, shape, dtype)

    def zeros(self, shape, dtype=np.float64):
        return DeviceArray(self, shape, dtype).zero()

    def to_device(self, arr, dtype=None):
        arr = np.asarray(arr)
        if dtype is None:
            dtype = arr.dtype
        return DeviceArray(self, arr.shape, dtype).upload(arr)

    # ---- kernels ---------------------------------------------------------------------
    def lqr_solve(self, dtype, T, B, n, m, x0, C, c, F, F_T, f, x, u, Ks, ks, fac=None,
                  flags=LQR_FACTOR | LQR_ROLLOUT, stream=None):
        self._check(self.lib.dmpc_lqr_solve(self.h, dtype_code(dtype), T, B, n, m, _p(x0), _p(C), _p(c), _p(F), F_T,
                                            _p(f), _p(x), _p(u), _p(Ks), _p(ks), _p(fac), flags, stream))

    def lqr_adjoint(self, dtype, T, B, n, m, C, c, F, x, u, gx, gu, Ks, fac, dx0, dC, dc, dF, df,
                    flags=ADJ_STRICT_REFERENCE, stream=None):
        self._check(self.lib.dmpc_lqr_adjoint(self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), _p(x), _p(u),
                                              _p(gx), _p(gu), _p(Ks), _p(fac), _p(dx0), _p(dC), _p(dc), _p(dF),
                                              _p(df), flags, stream))

    def lqr_shared_workspace_bytes(self, dtype, T, B, n, m, share=None):
        """share=None: the original entry point; an int (0 or SHARE_C): dmpc_lqr_shared_workspace_bytes_ex."""
        need = _sz(0)
        if share is None:
            self._check(self.lib.dmpc_lqr_shared_workspace_bytes(dtype_code(dtype), T, B, n, m, ctypes.byref(need)))
        else:
            self._check(self.lib.dmpc_lqr_shared_workspace_bytes_ex(dtype_code(dtype), T, B, n, m, int(share),
                                                                    ctypes.byref(need)))
        return int(need.value)

    def lqr_solve_shared(self, dtype, T, B, n, m, x0, C, c, F, F_T, f, x, u, ws, ws_bytes=None, stream=None, share=None):
        """C [T,s,s] and F [F_T,n,s] shared by the batch (and c [T,s] with share=SHARE_C); ws of
        lqr_shared_workspace_bytes(..., share) bytes.  share=None calls the original entry point."""
        ws_bytes = ws.nbytes if ws_bytes is None else ws_bytes
        a = (self.h, dtype_code(dtype), T, B, n, m, _p(x0), _p(C), _p(c), _p(F), int(F_T), _p(f), _p(x), _p(u), _p(ws),
             int(ws_bytes))
        if share is None:
            self._check(self.lib.dmpc_lqr_solve_shared(*a, stream))
        else:
            self._check(self.lib.dmpc_lqr_solve_shared_ex(*a, int(share), stream))

    def lqr_adjoint_shared(self, dtype, T, B, n, m, C, c, F, F_T, x, u, gx, gu, ws, dx0, dC, dc, dF, df,
                           flags=ADJ_STRICT_REFERENCE, ws_bytes=None, stream=None, share=None):
        """share=SHARE_C: c [T,s], dc [T,s] summed over the batch (or None).  share=None: the original entry point."""
        ws_bytes = ws.nbytes if ws_bytes is None else ws_bytes
        a = (self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), int(F_T), _p(x), _p(u), _p(gx), _p(gu), _p(ws),
             int(ws_bytes), _p(dx0), _p(dC), _p(dc), _p(dF), _p(df), flags)
        if share is None:
            self._check(self.lib.dmpc_lqr_adjoint_shared(*a, stream))
        else:
            self._check(self.lib.dmpc_lqr_adjoint_shared_ex(*a, int(share), stream))

    def pnqp(self, dtype, B, m, H, q, lower, upper, x_init, x, LU, piv, free, iters, flags=None, n_iter=20,
             coupling=COUPLING_ELEMENT, stream=None):
        self._check(self.lib.dmpc_pnqp(self.h, dtype_code(dtype), B, m, _p(H), _p(q), _p(lower), _p(upper), _p(x_init),
                                       n_iter, coupling, _p(x), _p(LU), _p(piv), _p(free), _p(iters), _p(flags), stream))

    @staticmethod
    def _dynp(params):
        arr = (ctypes.c_double * 5)(*([float(v) for v in params] + [0.0] * (5 - len(params)))) if params is not None else None
        return arr

    def mpc_step_forward(self, dtype, T, B, n, m, C, c, F, F_T, f, x_nom, u_nom, lower, upper, tC, tc, dynamics, tF,
                         tf, dyn_params, ls_decay, max_ls_trials, need_expand, coupling, x, u, Ks, ks, u_first, objs,
                         costs, old_costs, alphas, n_qp, free, n_ls, flags, stream=None):
        self._check(self.lib.dmpc_mpc_step_forward(
            self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), F_T, _p(f), _p(x_nom), _p(u_nom), _p(lower),
            _p(upper), _p(tC), _p(tc), dynamics, _p(tF), _p(tf), self._dynp(dyn_params), float(ls_decay),
            int(max_ls_trials), int(bool(need_expand)), coupling, _p(x), _p(u), _p(Ks), _p(ks), _p(u_first), _p(objs),
            _p(costs), _p(old_costs), _p(alphas), _p(n_qp), _p(free), _p(n_ls), _p(flags), stream))

    def mpc_step_backward(self, dtype, T, B, n, m, C, c, F, F_T, x, u, lower, upper, gx, gu, ws_Ks, ws_ks, ws_dtau,
                          active, dx0, dC, dc, dF, df, stream=None):
        self._check(self.lib.dmpc_mpc_step_backward(
            self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), F_T, _p(x), _p(u), _p(lower), _p(upper),
            _p(gx), _p(gu), _p(ws_Ks), _p(ws_ks), _p(ws_dtau), _p(active), _p(dx0), _p(dC), _p(dc), _p(dF), _p(df),
            stream))

    def lqr_active_solve(self, dtype, T, B, n, m, x0, C, c, F, F_T, f, active, x, u, Ks, ks, stream=None):
        self._check(self.lib.dmpc_lqr_active_solve(self.h, dtype_code(dtype), T, B, n, m, _p(x0), _p(C), _p(c), _p(F),
                                                   F_T, _p(f), _p(active), _p(x), _p(u), _p(Ks), _p(ks), stream))

    def get_traj(self, dtype, T, B, n, m, dynamics, x0, u, F, f, dyn_params, x, Fout=None, fout=None, stream=None):
        self._check(self.lib.dmpc_get_traj(self.h, dtype_code(dtype), T, B, n, m, dynamics, _p(x0), _p(u), _p(F), _p(f),
                                           self._dynp(dyn_params), _p(x), _p(Fout), _p(fout), stream))

    @staticmethod
    def split_reduced(sums, n, m):
        """(sum dC [s,s], sum dc [s], sum dF [n,s], sum df [n]) views of a dmpc_*_reduced result."""
        s = n + m
        o = 0
        out = []
        for shape in ((s, s), (s,), (n, s), (n,)):
            sz = int(np.prod(shape))
            out.append(sums[o:o + sz].reshape(shape))
            o += sz
        return tuple(out)

    def lqr_adjoint_reduced(self, dtype, T, B, n, m, C, c, F, x, u, gx, gu, Ks, fac, ws_dtau, ws_partials, dx0, sums,
                            flags=ADJ_STRICT_REFERENCE, stream=None):
        self._check(self.lib.dmpc_lqr_adjoint_reduced(
            self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), _p(x), _p(u), _p(gx), _p(gu), _p(Ks), _p(fac),
            _p(ws_dtau), _p(ws_partials), _p(dx0), _p(sums), flags, stream))

    def mpc_step_backward_reduced(self, dtype, T, B, n, m, C, c, F, F_T, x, u, lower, upper, gx, gu, ws_Ks, ws_ks,
                                  ws_dtau, active, ws_partials, dx0, sums, stream=None):
        self._check(self.lib.dmpc_mpc_step_backward_reduced(
            self.h, dtype_code(dtype), T, B, n, m, _p(C), _p(c), _p(F), F_T, _p(x), _p(u), _p(lower), _p(upper),
            _p(gx), _p(gu), _p(ws_Ks), _p(ws_ks), _p(ws_dtau), _p(active), _p(ws_partials), _p(dx0), _p(sums), stream))

    def expand_time_batch(self, dtype, T, B, src, dst, count, stream=None):
        """dst[t,b,:] = src[:] on the device (util.expand_time_batch, reference util.py:361-377)."""
        self._check(self.lib.dmpc_expand_time_batch(self.h, dtype_code(dtype), T, B, int(count), _p(src), _p(dst), stream))

    def reduced_grad_elems(self, n, m):
        return int(self.lib.dmpc_reduced_grad_elems(n, m))

    def warmstart_take(self, dtype, T, B, m, n_samples, cache, idx, u, stream=None):
        self._check(self.lib.dmpc_warmstart_take(self.h, dtype_code(dtype), T, B, m, n_samples, _p(cache), _p(idx), _p(u), stream))

    def warmstart_put(self, dtype, T, B, m, n_samples, cache, idx, u, stream=None):
        self._check(self.lib.dmpc_warmstart_put(self.h, dtype_code(dtype), T, B, m, n_samples, _p(cache), _p(idx), _p(u), stream))

    def boxddp_solve(self, dtype, T, B, n, m, x_init, C, c, lower, upper, dynamics, F, F_T, f, dyn_params, u_init,
                     eps, best_cost_eps, ls_decay, not_improved_lim, max_iter, max_ls_trials, coupling,
                     x_best, u_best, costs_best, du_best, du_last, F_lin=None, f_lin=None, stream=None, poll_every=0):
        """Device-resident BoxDDP loop; returns (n_iter, status, flags)."""
        need = _sz(0)
        self._check(self.lib.dmpc_boxddp_workspace_bytes(dtype_code(dtype), T, B, n, m, ctypes.byref(need)))
        ws = DeviceArray(self, (int(need.value),), np.uint8)
        opts = BoxDdpOpts(float(eps), float(best_cost_eps), float(ls_decay), int(not_improved_lim), int(max_iter),
                          int(max_ls_trials), int(coupling), int(poll_every))
        n_iter, status, flags = _i(0), _i(0), _i(0)
        try:
            self._check(self.lib.dmpc_boxddp_solve(
                self.h, dtype_code(dtype), T, B, n, m, _p(x_init), _p(C), _p(c), _p(lower), _p(upper), dynamics, _p(F),
                int(F_T), _p(f), self._dynp(dyn_params), _p(u_init), ctypes.cast(ctypes.byref(opts), _vp), _p(ws),
                int(need.value), _p(x_best), _p(u_best), _p(costs_best), _p(du_best), _p(du_last), _p(F_lin), _p(f_lin),
                ctypes.byref(n_iter), ctypes.byref(status), ctypes.byref(flags), stream))
        finally:
            ws.free()
        return int(n_iter.value), int(status.value), int(flags.value)

    def lqr_fac_elems(self, T, B, n, m):
        return int(self.lib.dmpc_lqr_fac_elems(T, B, n, m))


_default_ctx = {}


def default_context(device=0):
    """Process-wide context per device (created on first use; raises without a GPU)."""
    ctx = _default_ctx.get(device)
    if ctx is None:
        ctx = Context(device)
        _default_ctx[device] = ctx
    return ctx
