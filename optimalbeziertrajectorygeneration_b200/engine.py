"""Device-side engine behind the drop-in ``BezOptimization`` / ``Bezier`` API.

PyTorch is used only for device buffers, pinned staging buffers and streams;
all arithmetic happens in libbezgpu.so (hand-written sm_100a CUDA) reached
through the ctypes C-ABI in ``_capi``.  There is no CPU fallback.
"""
import ctypes

import numpy as np
import torch

from . import _capi, _tables

F64 = torch.float64


def _require_cuda():
    if not torch.cuda.is_available():
        raise _capi.BezGpuError(
            "no CUDA device visible: the Bezier constraint path runs only on the GPU "
            "(libbezgpu.so, sm_100a); there is no CPU fallback")


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream(device=None):
    """Raw handle of torch's current stream on ``device`` (default: the current device)."""
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_buffer(t, shape, what):
    """Caller-supplied device workspaces are handed to the kernels as raw pointers: a wrong
    size, dtype, layout or device would be an out-of-bounds device write."""
    if t is None:
        return
    if not isinstance(t, torch.Tensor) or t.dtype != F64 or not t.is_contiguous() or not t.is_cuda:
        raise ValueError("%s must be a contiguous float64 CUDA tensor" % what)
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s has shape %r, expected %r" % (what, tuple(t.shape), tuple(shape)))


class Plan:
    """Device-resident constant tables for one (degree, dim, DEG_ELEV).

    Replaces BezierParams.elevationMatrixCache / productMatrixCache
    (bezier.py:48-52): the tables are built once on the host with
    scipy.special.binom and live in HBM for the life of the plan."""

    _cache = {}

    def __init__(self, n, dim, elev, device):
        _require_cuda()
        self.n, self.dim, self.elev, self.device = int(n), int(dim), int(elev), int(device)
        self.L = 2 * self.n + self.elev + 1
        W = np.ascontiguousarray(_tables.prod_weights(self.n))
        T = np.ascontiguousarray(_tables.elev_matrix(2 * self.n, self.elev))
        E1 = np.ascontiguousarray(_tables.elev_matrix(self.n - 1, 1))
        handle = ctypes.c_void_p(0)
        _capi.call("bez_plan_create", self.n, self.dim, self.elev, self.device,
                   W.ctypes.data, T.ctypes.data, E1.ctypes.data, ctypes.byref(handle))
        self.handle = handle

    @classmethod
    def get(cls, n, dim, elev, device):
        key = (int(n), int(dim), int(elev), int(device))
        p = cls._cache.get(key)
        if p is None:
            p = cls._cache[key] = cls(*key)
        return p

    def __del__(self):
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            try:
                _capi.lib.bez_plan_destroy(h)
            except Exception:
                pass
            self.handle = None


class AngRateTables:
    """Device tables of the angular-rate kernel for one (degree, DEG_ELEV):
    elevMatrix(n,E), elevMatrix(m-1,1), C(m,.), C(2m,.) with m = n+E, all from
    scipy.special.binom like the reference's (bezier.py:1127-1147, 1183-1208)."""

    _cache = {}

    def __init__(self, n, elev, device):
        from scipy.special import binom
        _require_cuda()
        self.n, self.elev, self.m, self.device = int(n), int(elev), int(n + elev), int(device)
        m = self.m
        Tpos = np.ascontiguousarray(_tables.elev_matrix(self.n, self.elev))
        E1 = np.ascontiguousarray(_tables.elev_matrix(m - 1, 1))
        Cm = np.ascontiguousarray(binom(m, np.arange(m + 1)), dtype=np.float64)
        C2m = np.ascontiguousarray(binom(2 * m, np.arange(2 * m + 1)), dtype=np.float64)
        handle = ctypes.c_void_p(0)
        _capi.call("bez_angrate_tables_create", self.n, self.elev, self.device, Tpos.ctypes.data,
                   E1.ctypes.data, Cm.ctypes.data, C2m.ctypes.data, ctypes.byref(handle))
        self.handle = handle

    @classmethod
    def get(cls, n, elev, device):
        key = (int(n), int(elev), int(device))
        t = cls._cache.get(key)
        if t is None:
            t = cls._cache[key] = cls(*key)
        return t

    def __del__(self):
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            try:
                _capi.lib.bez_angrate_tables_destroy(h)
            except Exception:
                pass
            self.handle = None


def num_pairs(N):
    return N * (N - 1) // 2


def _on_device(method):
    """Runs an engine method with the engine's device current (entry points without a plan,
    torch allocations and stream lookups all follow the current device), so an engine built
    with ``device=k`` works whatever device the calling thread has selected."""
    import functools

    @functools.wraps(method)
    def wrapper(self, *a, **k):
        if torch.cuda.current_device() == self.dev_index:
            return method(self, *a, **k)
        with torch.cuda.device(self.device):
            return method(self, *a, **k)
    return wrapper


class ActiveSet:
    """Device destination of the reduced result of a fused kernel launch over ``nitems_total``
    flattened items (f = b * nitems + item): the packed bitmask ``mask`` (bit f & 31 of word
    f >> 5 = min < threshold) and, with ``capacity`` > 0, the compacted list ``idx[k]`` = f,
    ``val[k]`` = min of the active items (``count`` = how many there are; order unspecified;
    ``count`` > ``capacity`` means the list overflowed and only the mask is complete).
    All three live in ONE device buffer so that a single D2H copy brings the whole result:
    [count (8 B) | mask words | idx | val]."""

    def __init__(self, nitems_total, capacity, device, threshold=0.0):
        self.nitems_total = int(nitems_total)
        self.capacity = int(capacity)
        self.threshold = float(threshold)
        self.words = (self.nitems_total + 31) // 32
        self.mask_slots = (self.words + 1) // 2                 # 8-byte slots holding the mask
        self.nslots = 1 + self.mask_slots + 2 * self.capacity
        self.buf = torch.zeros(self.nslots, dtype=torch.int64, device=device)
        self.count = self.buf[0:1]
        self.mask = self.buf[1:1 + self.mask_slots].view(torch.int32)
        self.idx = self.buf[1 + self.mask_slots:1 + self.mask_slots + self.capacity]
        self.val = self.buf[1 + self.mask_slots + self.capacity:].view(F64)

    def check(self, nitems_total, device):
        if int(nitems_total) != self.nitems_total or self.buf.device != device:
            raise ValueError("ActiveSet was sized for %d items on %s" % (self.nitems_total, self.buf.device))

    def reset(self):
        """Zeroes the list counter (stream ordered; the mask is overwritten by the kernel)."""
        self.count.zero_()

    @staticmethod
    def decode(host_buf, nitems_total, capacity):
        """host copy of ``buf`` (int64 numpy array) -> (flags bool [nitems_total], idx, val,
        overflow): idx / val sorted by idx."""
        words = (nitems_total + 31) // 32
        slots = (words + 1) // 2
        count = int(host_buf[0])
        mask = host_buf[1:1 + slots].view(np.uint32)[:words]
        flags = np.unpackbits(mask.view(np.uint8), bitorder='little')[:nitems_total].astype(bool)
        k = min(count, capacity)
        idx = host_buf[1 + slots:1 + slots + k]
        val = host_buf[1 + slots + capacity:1 + slots + capacity + k].view(np.float64)
        order = np.argsort(idx, kind='stable')
        return flags, idx[order], val[order], count > capacity


class ConstraintEngine:
    """Everything a BezOptimization model needs on the device.

    ``model`` is the reference's model dict (optimization.py:49-63);
    ``point_obstacles`` the list handed to the constructor."""

    def __init__(self, model, point_obstacles=None, device=None):
        _require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.dev_index = self.device.index
        self.numVeh = int(model['numVeh'])
        self.dim = int(model['dim'])
        self.n = int(model['deg'])
        self.timeopt = model['minGoal'].lower() == 'timeopt'
        self.tf_fixed = float(model['tf'])
        init = model['initPoints']
        self.fixed_ends = init is not None and init.dtype != object
        ispd = model['initSpeeds']
        self.dubins = ispd[0] is not None
        self.offset = (1 if self.fixed_ends else 0) + (1 if self.dubins else 0)
        self.ncols = self.n + 1 - 2 * self.offset
        self.nvar = self.numVeh * self.dim * self.ncols + (1 if self.timeopt else 0)
        obst = None if point_obstacles is None else np.asarray(point_obstacles, dtype=np.float64)
        self.nObs = 0 if obst is None else int(obst.shape[0])
        self.N = self.numVeh + self.nObs
        self.row_stride = (self.dim * (self.n + 1) + 1) // 2 * 2

        def dev(a):
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.device)

        self.d_init = dev(init) if self.fixed_ends else None
        self.d_final = dev(model['finalPoints']) if self.fixed_ends else None
        if self.dubins:
            ia = np.asarray(model['initAngs'], dtype=np.float64)
            fa = np.asarray(model['finalAngs'], dtype=np.float64)
            self.d_ispeed = dev(np.asarray(ispd, dtype=np.float64))
            self.d_fspeed = dev(np.asarray(model['finalSpeeds'], dtype=np.float64))
            self.d_icos, self.d_isin = dev(np.cos(ia)), dev(np.sin(ia))
            self.d_fcos, self.d_fsin = dev(np.cos(fa)), dev(np.sin(fa))
        else:
            self.d_ispeed = self.d_fspeed = self.d_icos = self.d_isin = self.d_fcos = self.d_fsin = None
        self.d_obst = dev(obst[:, :self.dim]) if self.nObs else None
        self._pinned = {}
        self._x_stage = [None, None]        # rotating pinned staging buffers of upload()
        self._x_event = [None, None]
        self._x_turn = 0

    def _st(self):
        """Launch stream: torch's current stream on the engine's own device."""
        return _stream(self.device)

    def _check(self, t, shape, what):
        _check_buffer(t, shape, what)
        if t is not None and t.device != self.device:
            raise ValueError("%s lives on %s, the engine on %s" % (what, t.device, self.device))

    # -- plans -----------------------------------------------------------
    def plan(self, elev):
        return Plan.get(self.n, self.dim, elev, self.dev_index)

    # -- host <-> device staging ----------------------------------------
    def _pinned_buf(self, key, numel):
        buf = self._pinned.get(key)
        if buf is None or buf.numel() < numel:
            buf = torch.empty(max(numel, 1), dtype=F64, pin_memory=True)
            self._pinned[key] = buf
        return buf[:numel]

    def _pinned_buf_i64(self, key, numel):
        buf = self._pinned.get(key)
        if buf is None or buf.numel() < numel:
            buf = torch.empty(max(numel, 1), dtype=torch.int64, pin_memory=True)
            self._pinned[key] = buf
        return buf[:numel]

    @_on_device
    def upload(self, X):
        """host float64 [B, nvar] -> device tensor, through pinned memory."""
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        if X.shape[1] != self.nvar:
            raise ValueError("x has %d entries, the model expects %d" % (X.shape[1], self.nvar))
        # two staging buffers in rotation; a buffer is rewritten only after the H2D copy that
        # last read it has completed (event), so back-to-back uploads never race an in-flight DMA
        i = self._x_turn
        self._x_turn ^= 1
        if self._x_event[i] is not None:
            self._x_event[i].synchronize()
        stage = self._x_stage[i]
        if stage is None or stage.numel() < X.size:
            stage = self._x_stage[i] = torch.empty(max(X.size, 1), dtype=F64, pin_memory=True)
        stage = stage[:X.size]
        stage.numpy()[:] = X.ravel()
        d = torch.empty(X.shape, dtype=F64, device=self.device)
        st = torch.cuda.current_stream(self.device)
        with torch.cuda.stream(st):
            d.view(-1).copy_(stage, non_blocking=True)
            ev = self._x_event[i] = torch.cuda.Event()
            ev.record(st)
        return d

    @_on_device
    def download(self, t, key="out", copy=True):
        """device tensor -> host numpy array (one sync).  With copy=False the
        returned array aliases the pinned staging buffer named ``key`` and is only valid
        until the next download with the same key (the closures of BezOptimization use
        one key each, so results of different closures never alias)."""
        stage = self._pinned_buf(key, t.numel())
        st = torch.cuda.current_stream(self.device)
        with torch.cuda.stream(st):
            stage.copy_(t.reshape(-1), non_blocking=True)
        st.synchronize()
        host = stage.numpy().reshape(tuple(t.shape))
        return host.copy() if copy else host

    # -- A0 -----------------------------------------------------------------
    @_on_device
    def assemble(self, d_x, elev=0, obst_sets=None, evals_per_set=0):
        """reshapeVector (+ obstacle rows) for every row of d_x [B, nvar].
        Returns (cpts [B, N, S], tf [B]) with S = dim*(n+1) rounded up to even.
        ``obst_sets`` [nsets, nObs, dim] (device) with ``evals_per_set`` > 0: row b takes the
        obstacles of set b // evals_per_set (batches of independent problems, batch.py)."""
        B = int(d_x.shape[0])
        plan = self.plan(elev)
        cpts = torch.empty((B, self.N, self.row_stride), dtype=F64, device=self.device)
        tf = torch.empty((B,), dtype=F64, device=self.device)
        if obst_sets is not None:
            if tuple(obst_sets.shape[1:]) != (self.nObs, self.dim) or evals_per_set <= 0 or \
                    int(obst_sets.shape[0]) * evals_per_set < B:
                raise ValueError("obstacle sets do not cover the %d evaluation points" % B)
        _capi.call("bez_assemble_cpts_sets", plan.handle, _ptr(d_x), B, self.nvar, self.numVeh, self.nObs,
                   int(self.fixed_ends), int(self.dubins), int(self.timeopt), self.tf_fixed,
                   _ptr(self.d_init), _ptr(self.d_final), _ptr(self.d_ispeed), _ptr(self.d_fspeed),
                   _ptr(self.d_icos), _ptr(self.d_isin), _ptr(self.d_fcos), _ptr(self.d_fsin),
                   _ptr(self.d_obst if obst_sets is None else obst_sets),
                   int(evals_per_set) if obst_sets is not None else 0, _ptr(cpts), _ptr(tf), self._st())
        return cpts, tf

    # -- A1-A4 --------------------------------------------------------------
    def _reduce_opts(self, B, nitems, itemmin, min_pitch, peer_ptrs, active):
        """ctypes bez_reduce_opts (+ the objects that must outlive the call)."""
        o = _capi.ReduceOpts()
        keep = []
        if itemmin is not None:
            o.itemmin = itemmin.data_ptr()
        o.min_pitch = int(min_pitch or 0)
        if peer_ptrs:
            arr = (ctypes.c_uint64 * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
            keep.append(arr)
            o.peer_min = ctypes.addressof(arr)
            o.npeers = len(peer_ptrs)
        if active is not None:
            active.check(B * nitems, self.device)
            o.active_mask = active.mask.data_ptr()
            o.threshold = float(active.threshold)
            if active.capacity > 0:
                o.list_count = active.count.data_ptr()
                o.list_idx = active.idx.data_ptr()
                o.list_val = active.val.data_ptr()
                o.list_cap = int(active.capacity)
        return o, keep

    @_on_device
    def separation(self, cpts, elev, max_sep, pair_begin=0, npairs=None, out=None, pairmin=None,
                   n_curves=None, peer_ptrs=None, rows=True, min_pitch=None, active=None):
        """Fused sub -> normSquare -> elev -> -maxSep^2 over a range of the
        lexicographic pair list.  Returns out [B, npairs, L] (device).
        ``pairmin`` [B, npairs] (or, with ``min_pitch``, a view of a wider [B, min_pitch] matrix
        starting at this range's first column): min over each pair's L values.
        ``peer_ptrs``: device addresses in other GPUs' gathered per-pair-minimum matrices
        (sharding.PeerMinima); the kernel then also stores every minimum there over NVLink.
        ``active``: an :class:`ActiveSet` that receives the packed bitmask / compacted list of
        the pairs with minimum < threshold.  ``rows=False``: no rows are written (returns None)."""
        plan = self.plan(elev)
        B = int(cpts.shape[0])
        N = int(cpts.shape[1]) if n_curves is None else int(n_curves)
        if npairs is None:
            npairs = num_pairs(N) - pair_begin
        if pair_begin < 0 or npairs < 0 or pair_begin + npairs > num_pairs(N):
            raise ValueError("pair range [%d, %d) outside the %d pairs" % (pair_begin, pair_begin + npairs, num_pairs(N)))
        self._check(cpts, (B, int(cpts.shape[1]), self.row_stride), "cpts")
        if rows:
            if out is None:
                out = torch.empty((B, npairs, plan.L), dtype=F64, device=self.device)
            self._check(out, (B, npairs, plan.L), "out")
        else:
            out = None
            if pairmin is None and active is None and not peer_ptrs:
                raise ValueError("rows=False needs pairmin, active or peer_ptrs")
        if min_pitch:
            if pairmin is None or int(min_pitch) < npairs:
                raise ValueError("min_pitch needs pairmin and must be >= npairs")
            if pairmin.dtype != F64 or pairmin.device != self.device or pairmin.stride(-1) != 1 or \
                    (B > 1 and pairmin.stride(0) != int(min_pitch)) or pairmin.shape[0] != B or pairmin.shape[1] < npairs:
                raise ValueError("pairmin must be a float64 view [B, >= npairs] with row pitch min_pitch")
        else:
            self._check(pairmin, (B, npairs), "pairmin")
        if peer_ptrs and pairmin is None:
            raise ValueError("peer_ptrs needs the local pairmin destination")
        if peer_ptrs and not min_pitch and (pair_begin != 0 or npairs != num_pairs(N)):
            # the kernel addresses the peers' matrices with the same pitch as the local one:
            # a sub-range needs min_pitch (and pointers offset to the range's first column)
            raise ValueError("peer_ptrs with a pair sub-range needs min_pitch")
        opts, keep = self._reduce_opts(B, npairs, pairmin, min_pitch, peer_ptrs, active)
        _capi.call("bez_pair_sepsq_elev_ex", plan.handle, _ptr(cpts), B, N, int(pair_begin), int(npairs),
                   float(max_sep) ** 2, _ptr(out), ctypes.byref(opts), self._st())
        del keep
        return out

    # -- A5 -------------------------------------------------------------------
    @_on_device
    def speed(self, cpts, tf, elev, alpha, beta, veh_begin=0, nveh=None, out=None, vehmin=None, active=None):
        """alpha * (squared speed control points) + beta, [B, nveh, L]; ``vehmin`` [B, nveh]
        receives the minimum over each vehicle's L values, ``active`` its bitmask / list."""
        plan = self.plan(elev)
        B = int(cpts.shape[0])
        N = int(cpts.shape[1])
        if nveh is None:
            nveh = self.numVeh - veh_begin
        if out is None:
            out = torch.empty((B, nveh, plan.L), dtype=F64, device=self.device)
        self._check(cpts, (B, N, self.row_stride), "cpts")
        self._check(tf, (B,), "tf")
        self._check(out, (B, nveh, plan.L), "out")
        self._check(vehmin, (B, nveh), "vehmin")
        if active is not None and vehmin is None:
            vehmin = torch.empty((B, nveh), dtype=F64, device=self.device)
        opts, keep = self._reduce_opts(B, nveh, vehmin, None, None, active)
        _capi.call("bez_speed_sq_elev_ex", plan.handle, _ptr(cpts), _ptr(tf), B, N, int(veh_begin),
                   int(nveh), float(alpha), float(beta), _ptr(out), ctypes.byref(opts), self._st())
        del keep
        return out

    # -- A6 -------------------------------------------------------------------
    @_on_device
    def angrate(self, cpts, tf, elev, alpha, beta, veh_begin=0, nveh=None, out=None):
        """alpha * (squared angular rate control points) + beta, [B, nveh, 4(n+E)+1]."""
        if self.dim != 2:
            raise ValueError('The input curve must be two dimensional,\n'
                             'instead it is {} dimensional'.format(self.dim))
        tabs = AngRateTables.get(self.n, elev, self.dev_index)
        B, N = int(cpts.shape[0]), int(cpts.shape[1])
        if nveh is None:
            nveh = self.numVeh - veh_begin
        L4 = 4 * (self.n + int(elev)) + 1
        if out is None:
            out = torch.empty((B, nveh, L4), dtype=F64, device=self.device)
        self._check(cpts, (B, N, self.row_stride), "cpts")
        self._check(tf, (B,), "tf")
        self._check(out, (B, nveh, L4), "out")
        _capi.call("bez_angrate_sq", tabs.handle, _ptr(cpts), _ptr(tf), B, N, self.row_stride,
                   int(veh_begin), int(nveh), float(alpha), float(beta), _ptr(out), self._st())
        return out

    # -- A7 ---------------------------------------------------------------------
    @staticmethod
    def fd_steps(x0, abs_step=1.4901161193847656e-08):
        """h and dx = (x0+h)-x0 exactly as SciPy's approx_derivative chooses them
        for SLSQP (scipy/optimize/_numdiff.py:585-596; abs_step = sqrt(eps) from
        _slsqp_py.py).  Host logic."""
        x0 = np.asarray(x0, dtype=np.float64)
        h = np.full_like(x0, abs_step)
        dx = (x0 + h) - x0
        sign = (x0 >= 0).astype(np.float64) * 2 - 1
        h = np.where(dx == 0, np.finfo(np.float64).eps ** 0.5 * sign * np.maximum(1.0, np.abs(x0)), h)
        return h, (x0 + h) - x0

    def _direction_rows(self):
        """d(control points)/d tf for time-optimal Dubins models: only control
        points 1 and n-1 depend on tf (optimization.py:273-281)."""
        if not (self.timeopt and self.dubins):
            return None
        if getattr(self, "_dir", None) is None:
            D = torch.zeros((self.N, self.row_stride), dtype=F64, device=self.device)
            nc = self.n + 1
            cs_i = (self.d_icos, self.d_isin)
            cs_f = (self.d_fcos, self.d_fsin)
            for d in range(2):
                D[:self.numVeh, d * nc + 1] += self.d_ispeed * cs_i[d] / self.n
                D[:self.numVeh, d * nc + self.n - 1] -= self.d_fspeed * cs_f[d] / self.n
            self._dir = D
        return self._dir

    @staticmethod
    def _fd_steps_device(d_x, abs_step=1.4901161193847656e-08):
        """dx of :meth:`fd_steps` for a device tensor (the same IEEE operations)."""
        h = torch.full_like(d_x, abs_step)
        dx = (d_x + h) - d_x
        sign = (d_x >= 0).to(F64) * 2 - 1
        rel = sign * torch.clamp(d_x.abs(), min=1.0) * np.finfo(np.float64).eps ** 0.5
        h = torch.where(dx == 0, rel, h)
        return (d_x + h) - d_x

    @_on_device
    def _fd_base(self, x, elev, obst_sets=None):
        """The base points of the closed-form Jacobians: ``x`` [nvar] or [B, nvar], host or device
        -> (cpts [B, N, S], tf [B], SciPy's divisors dx [B, nvar], batched = x is 2-D), the tuple
        their ``base=`` takes.  ``obst_sets`` [B, nObs, dim] (device): point b's own obstacles."""
        on_device = isinstance(x, torch.Tensor)
        x = x if on_device else np.asarray(x, dtype=np.float64)
        if x.ndim not in (1, 2) or int(x.shape[-1]) != self.nvar:
            raise ValueError("x must be [%d] or [B, %d]" % (self.nvar, self.nvar))
        if on_device:
            d_x = x.to(device=self.device, dtype=F64).reshape(-1, self.nvar).contiguous()
            d_dx = self._fd_steps_device(d_x)
        else:
            x2 = np.atleast_2d(x)
            d_x = self.upload(x2)
            d_dx = torch.as_tensor(self.fd_steps(x2)[1], device=self.device)
        cpts, tf = self.assemble(d_x, elev, obst_sets=obst_sets, evals_per_set=1 if obst_sets is not None else 0)
        return cpts, tf, d_dx, x.ndim == 2

    def _jac_out(self, out, shape, batched):
        """Destination [B, rows, cols] of a closed-form Jacobian (``out`` or a new tensor), viewed
        without the leading B for a 1-D x; a caller's ``out`` has x's rank."""
        if out is None:
            out = torch.empty(shape, dtype=F64, device=self.device)
        else:
            self._check(out, shape if batched else shape[1:], "out")
        return out if batched else out.view(shape[1:])

    @_on_device
    def jac_separation(self, x, elev, dense=True, out=None, obst_sets=None, npairs=None, base=None):
        """SciPy's 2-point Jacobian of the separation block in closed form (bez_jac_sepsq_elev_batched).
        ``x`` [nvar] or [B, nvar], host or device; ``obst_sets`` [B, nObs, dim] (device): point b's
        own obstacles (problem batches); ``npairs``: the leading pairs that get rows (default all;
        at least every pair with a vehicle).
        dense: J^T [B, nvar, npairs*L]; else the sweep layout
        [B, numVeh*dim*ncols*(N-1) + (npairs if time-optimal), L]; without the leading B for 1-D x.
        ``out``: the destination, in either layout and x's rank.
        ``base``: :meth:`_fd_base` of x already at hand (ProblemBatch.sweep); x is then ignored."""
        plan = self.plan(elev)
        cpts, _, d_dx, batched = self._fd_base(x, elev, obst_sets) if base is None else base
        B, L = int(cpts.shape[0]), plan.L
        npairs = num_pairs(self.N) if npairs is None else int(npairs)
        kdir = self.nvar - 1 if self.timeopt else -1
        if dense:
            shape = (B, self.nvar, npairs * L)
        else:
            shape = (B, self.numVeh * self.dim * self.ncols * (self.N - 1) + (npairs if self.timeopt else 0), L)
        out = self._jac_out(out, shape, batched)
        _capi.call("bez_jac_sepsq_elev_batched", plan.handle, _ptr(cpts), B, self.N, self.numVeh, self.ncols,
                   self.offset, _ptr(d_dx), _ptr(self._direction_rows()), kdir, npairs, int(bool(dense)), _ptr(out),
                   npairs * L if dense else 0, self._st())
        return out

    @_on_device
    def jac_speed(self, x, elev, alpha, dense=True, out=None, base=None):
        """SciPy's 2-point Jacobian of the speed block alpha * (squared speed) + beta in closed form
        (bez_jac_speed_sq_elev_batched); tf of each point from assemble.  ``x``, ``out``, ``base``
        as in :meth:`jac_separation`.
        dense: J^T [B, nvar, numVeh*L]; else [B, numVeh*dim*ncols + (numVeh if time-optimal), L];
        without the leading B for 1-D x."""
        plan = self.plan(elev)
        cpts, tf, d_dx, batched = self._fd_base(x, elev) if base is None else base
        B, L = int(cpts.shape[0]), plan.L
        kdir = self.nvar - 1 if self.timeopt else -1
        if dense:
            shape = (B, self.nvar, self.numVeh * L)
        else:
            shape = (B, self.numVeh * self.dim * self.ncols + (self.numVeh if self.timeopt else 0), L)
        out = self._jac_out(out, shape, batched)
        _capi.call("bez_jac_speed_sq_elev_batched", plan.handle, _ptr(cpts), _ptr(tf), B, int(cpts.shape[1]),
                   self.numVeh, self.ncols, self.offset, float(alpha), _ptr(d_dx), _ptr(self._direction_rows()),
                   kdir, int(bool(dense)), _ptr(out), self.numVeh * L if dense else 0, self._st())
        return out

    @_on_device
    def fd_points(self, X):
        """host X [B, nvar] -> device (Xp [B, nvar+1, nvar], dx [B, nvar]): the base point and the
        nvar forward points of every row, h and dx as SciPy chooses them (:meth:`fd_steps`)."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        B, n = X.shape[0], self.nvar
        h, dx = self.fd_steps(X)
        d_x, d_xh, d_dx = self.upload(np.concatenate((X, X + h, dx))).split(B)     # one pinned H2D
        Xp = d_x[:, None, :].repeat(1, n + 1, 1)
        Xp.view(B, -1)[:, n::n + 1] = d_xh          # forward point k+1 moves x_k: entry (k+1)*n + k
        return Xp, d_dx

    @_on_device
    def fd_quotient(self, F, dx):
        """SciPy's 2-point quotient of B sweeps (bez_fd_quotient_batched): F [B, nvar+1, m] holds
        f at the base point and the nvar forward points of :meth:`fd_points`, dx [B, nvar] ->
        J^T [B, nvar, m]."""
        B, m = int(dx.shape[0]), int(F.shape[-1])
        self._check(F, (B, self.nvar + 1, m), "F")
        self._check(dx, (B, self.nvar), "dx")
        JT = torch.empty((B, self.nvar, m), dtype=F64, device=self.device)
        _capi.call("bez_fd_quotient_batched", _ptr(F), _ptr(dx), B, self.nvar, m, _ptr(JT), self._st())
        return JT

    @_on_device
    def jac_angrate(self, x, elev, alpha, beta):
        """Literal '2-point' FD Jacobian of the angular-rate block: base point and
        all nvar perturbed points are evaluated in one batched launch (what SciPy
        does serially with the reference), then differenced on the device.
        Returns J^T [nvar, numVeh*(4m+1)]."""
        Xp, dx = self.fd_points(x)
        cpts, tf = self.assemble(Xp.view(-1, self.nvar), elev)
        F = self.angrate(cpts, tf, elev, alpha, beta).view(1, self.nvar + 1, -1)
        return self.fd_quotient(F, dx)[0]

    @_on_device
    def jac_angrate_closed(self, x, elev, alpha, dense=True, out=None, base=None):
        """Closed-form '2-point' Jacobian of the angular-rate block (bez_jac_angrate_sq): SciPy's
        quotient for the row alpha * (squared angular rate) + beta, without evaluating the
        perturbed points.  ``x``, ``out``, ``base`` as in :meth:`jac_separation` (the vehicle rows
        of a base with obstacles serve as well).
        dense: J^T [B, nvar, numVeh*(4m+1)]; else the sweep layout
        [B, numVeh*2*ncols + (numVeh if time-optimal), 4m+1]; without the leading B for 1-D x.
        n + elev > 127 raises BezGpuError (jac_angrate covers those shapes)."""
        if self.dim != 2:
            raise ValueError('The input curve must be two dimensional,\n'
                             'instead it is {} dimensional'.format(self.dim))
        tabs = AngRateTables.get(self.n, elev, self.dev_index)
        cpts, tf, d_dx, batched = self._fd_base(x, elev) if base is None else base
        B = int(cpts.shape[0])
        kdir = self.nvar - 1 if self.timeopt else -1
        L4 = 4 * (self.n + int(elev)) + 1
        if dense:
            shape = (B, self.nvar, self.numVeh * L4)
        else:
            shape = (B, self.numVeh * 2 * self.ncols + (self.numVeh if self.timeopt else 0), L4)
        out = self._jac_out(out, shape, batched)
        nscr = int(_capi.lib.bez_jac_angrate_scratch_doubles(B, self.numVeh, self.n, int(elev)))
        key = ("jac_angrate_scratch", nscr)
        scratch = getattr(self, "_scratch", {}).get(key)
        if scratch is None:
            scratch = torch.empty(max(nscr, 1), dtype=F64, device=self.device)
            self._scratch = {key: scratch}                 # one cached buffer per engine
        _capi.call("bez_jac_angrate_sq", tabs.handle, _ptr(cpts), _ptr(tf), B, int(cpts.shape[1]), self.row_stride,
                   self.numVeh, self.ncols, self.offset, self.nvar, _ptr(d_dx), _ptr(self._direction_rows()), kdir,
                   float(alpha), int(bool(dense)), _ptr(scratch), _ptr(out), shape[2], self._st())
        return out
