"""Drop-in mirror of the reference's ``optimization.py`` whose constraint and
cost callables run on the B200 (libbezgpu.so) instead of numpy/numba.

Same names, argument meaning and error behaviour as the reference:
``BezOptimization(numVeh, dimension, degree, minimizeGoal, maxSep, minSpeed,
maxSpeed, maxAngRate, initPoints, finalPoints, initSpeeds, finalSpeeds,
initAngs, finalAngs, tf, pointObstacles, shapeObstacles)`` with *properties
returning closures* ``f(x: float64[nvar]) -> float64[m]`` that are handed to
``scipy.optimize.minimize(method='SLSQP')`` (optimization.py:20-187), the module
global ``DEG_ELEV`` that is re-read at call time (optimization.py:17, SURVEY Q9),
``generateGuess`` and ``reshapeVector``.

Additive API (not in the reference): ``*_jac`` closures returning the
finite-difference Jacobian SciPy would have formed with nvar+1 calls, computed
in one batched launch; ``evaluate_batch`` for device-resident batched
evaluation.
"""
import numpy as np
import torch

from . import engine as _engine

DEG_ELEV = 0


def _on_model_device(method):
    """Runs a method with the model's device current (a model built with ``device=k`` works
    whatever device the calling thread has selected; the caller's device is restored)."""
    import functools

    @functools.wraps(method)
    def wrapper(self, *a, **k):
        if self._device is None or not torch.cuda.is_available() or torch.cuda.current_device() == self._device:
            return method(self, *a, **k)
        with torch.cuda.device(self._device):
            return method(self, *a, **k)
    return wrapper


def _deg_elev():
    # re-read the module global at call time, like the reference (Q9)
    return int(globals()['DEG_ELEV'])


class SweepActive:
    """Host-side (pinned, reused by the next call) reduced result of
    :meth:`BezOptimization.evaluate_sweep_active`: per chunk of evaluations the packed
    active-pair bitmask + compacted (pair, min) list, and the max-speed minima per vehicle."""

    def __init__(self, pair_bufs, veh_bufs, vehmin, M, chunk, P, nv, cap):
        self.pair_bufs, self.veh_bufs, self.vehmin = pair_bufs, veh_bufs, vehmin
        self.M, self.chunk, self.P, self.nv, self.cap = M, chunk, P, nv, cap
        self.nchunks = pair_bufs.shape[0]
        self.overrides = {}

    def rows_of(self, k):
        return min(self.chunk, self.M - k * self.chunk)

    def pair_counts(self):
        """number of active pairs per chunk (from the list counters)"""
        return self.pair_bufs[:, 0].copy()

    def pairs(self, k):
        """chunk k -> (flags bool [b, P], eval index [m], pair index [m], minimum [m]) of the
        active pairs, sorted by (eval, pair)."""
        b = self.rows_of(k)
        if k in self.overrides:
            flags, idx, val, over = _engine.ActiveSet.decode(self.overrides[k], b * self.P, b * self.P)
        else:
            flags, idx, val, over = _engine.ActiveSet.decode(self.pair_bufs[k], b * self.P, self.cap)
        assert not over
        return flags.reshape(b, self.P), idx // self.P, idx % self.P, val

    def vehicles(self, k):
        """chunk k -> (minimum of the max-speed block per vehicle [b, nv], flags [b, nv])"""
        b = self.rows_of(k)
        flags, _, _, _ = _engine.ActiveSet.decode(self.veh_bufs[k], b * self.nv, 0)
        lo = k * self.chunk
        return self.vehmin[lo:lo + b], flags.reshape(b, self.nv)


class BezOptimization:
    def __init__(self,
                 numVeh=1,
                 dimension=1,
                 degree=5,
                 minimizeGoal='Euclidean',
                 maxSep=0.9,
                 minSpeed=0,
                 maxSpeed=1e6,
                 maxAngRate=1e6,
                 initPoints=None,
                 finalPoints=None,
                 initSpeeds=None,
                 finalSpeeds=None,
                 initAngs=None,
                 finalAngs=None,
                 tf=1.0,
                 pointObstacles=None,
                 shapeObstacles=None,
                 device=None):
        self.pointObstacles = pointObstacles
        self.shapeObstacles = shapeObstacles

        self._numCols = degree + 1
        if initPoints is not None:
            self._numCols -= 2
        if initSpeeds is not None:
            self._numCols -= 2

        # optimization.py:49-63
        self.model = {'numVeh': numVeh,
                      'dim': dimension,
                      'deg': degree,
                      'minGoal': minimizeGoal,
                      'maxSep': maxSep,
                      'minSpeed': minSpeed,
                      'maxSpeed': maxSpeed,
                      'maxAngRate': maxAngRate,
                      'initPoints': np.atleast_2d(initPoints),
                      'finalPoints': np.atleast_2d(finalPoints),
                      'initSpeeds': np.atleast_1d(initSpeeds),
                      'finalSpeeds': np.atleast_1d(finalSpeeds),
                      'initAngs': np.atleast_1d(initAngs),
                      'finalAngs': np.atleast_1d(finalAngs),
                      'tf': tf}
        self._device = device
        # additive: when True the closures return views of a pinned staging buffer
        # (one buffer per closure: valid until the next call of the *same* closure)
        # instead of copies
        self.zero_copy_results = False
        self._engines = {}

    # ------------------------------------------------------------------
    def _model_signature(self):
        """What the device state was built from.  The reference re-reads ``model`` and
        ``pointObstacles`` on every call; here the engine is rebuilt when an entry is
        *replaced* (identity / scalar value changes).  In-place edits of the arrays inside
        are not seen: call :meth:`invalidate` after those."""
        m = self.model
        po = self.pointObstacles
        return (m['numVeh'], m['dim'], m['deg'], str(m['minGoal']).lower(), float(m['tf']),
                id(m['initPoints']), id(m['finalPoints']), id(m['initSpeeds']), id(m['finalSpeeds']),
                id(m['initAngs']), id(m['finalAngs']), id(po), None if po is None else len(po))

    def invalidate(self):
        """Drops the cached device state (after in-place edits of model arrays / obstacles)."""
        self._engines = {}

    def _engine(self, with_obstacles):
        """Device state; built lazily so constructing a model needs no GPU."""
        key = bool(with_obstacles) and self.pointObstacles is not None
        sig = self._model_signature()
        if getattr(self, '_engines_sig', None) != sig:
            self._engines, self._engines_sig = {}, sig
        eng = self._engines.get(key)
        if eng is None:
            eng = _engine.ConstraintEngine(self.model, self.pointObstacles if key else None,
                                           device=self._device)
            self._engines[key] = eng
        return eng

    @property
    def nvar(self):
        return (self.model['numVeh'] * self.model['dim'] * self._numCols +
                (1 if self.model['minGoal'].lower() == 'timeopt' else 0))

    # ------------------------------------------------------------------
    @property
    def objectiveFunction(self):
        minGoal = self.model['minGoal'].lower()

        objectivesDict = {'euclidean': self.euclideanObjective,
                          'timeopt': lambda x: x[-1],
                          'accel': self.accelObjective,
                          'jerk': self.jerkObjective,
                          }
        try:
            return objectivesDict[minGoal]
        except KeyError:
            err = ('The provided minimize goal, {}, is not a valid goal. '
                   'The available minimize goals are:\n{}'
                   ).format(minGoal, objectivesDict.keys())
            raise ValueError(err)

    # ------------------------------------------------------------------
    @property
    def temporalSeparationConstraints(self):
        """optimization.py:83-107 -> _temporalSeparationConstraints (:311-346)."""
        def wrapper(x):
            eng = self._engine(with_obstacles=True)
            if eng.N <= 1:
                return None                       # optimization.py:345-346
            E = _deg_elev()
            cpts, _ = eng.assemble(eng.upload(x), E)
            out = eng.separation(cpts, E, self.model['maxSep'])
            return eng.download(out, key="out:sep", copy=not self.zero_copy_results).reshape(-1)
        return wrapper

    # -- A13 ---------------------------------------------------------------
    # Budgets of the bounded branch-and-bound (the reference recurses without bound, Q6) and
    # what to do with a pair that exhausts them: 'raise' (default) raises RecursionError, which
    # is what the reference does on such a pair under Python's default recursion limit;
    # 'nan' returns NaN rows and leaves the per-pair status in ``last_status``.
    spatial_max_depth = 200
    spatial_max_nodes = 1 << 18
    spatial_on_limit = 'raise'

    def _spatial_shapes(self):
        """Shape obstacles as arrays: ('curve', cpts [dim, n+1]) for Bezier objects (what the
        reference accepts) and, additively, ('poly', vertices [m, 3]) for convex polytopes
        given as [m, 2 or 3] vertex arrays (routed through minDist2Poly, bezier.py:1411-1496)."""
        shapes = []
        for obstacle in (self.shapeObstacles or []):
            if hasattr(obstacle, 'cpts'):
                shapes.append(('curve', np.ascontiguousarray(obstacle.cpts, dtype=np.float64)))
            else:
                v = np.asarray(obstacle, dtype=np.float64)
                if v.ndim != 2 or v.shape[1] not in (2, 3):
                    raise TypeError('shape obstacles must be Bezier curves or [m, 2|3] vertex arrays')
                if v.shape[1] == 2:
                    v = np.hstack([v, np.zeros((v.shape[0], 1))])
                shapes.append(('poly', np.ascontiguousarray(v)))
        return shapes

    def _spatial_rows(self, Y):
        """Y [B, numVeh*dim, deg+1] control-point matrices -> (rows [B, npairs, 3], status
        [B, npairs]): minDist of every pair i<j among vehicles + shape obstacles, one launch per
        group of pairs of equal (kind, shape) -- mixed degrees / dimensions and polytopes form
        their own groups.  Pairs that do not contain a vehicle are computed for b = 0 only."""
        from . import bezier as _bez
        numVeh, dim = self.model['numVeh'], self.model['dim']
        B = Y.shape[0]
        shapes = self._spatial_shapes()
        nobj = numVeh + len(shapes)
        pairs = [(i, j) for i in range(nobj) for j in range(i + 1, nobj)]
        rows = np.empty((B, len(pairs), 3))
        status = np.zeros((B, len(pairs)), dtype=np.int32)

        def obj(b, i):
            if i < numVeh:
                return 'curve', np.ascontiguousarray(Y[b, i * dim:(i + 1) * dim, :])
            return shapes[i - numVeh]

        groups = {}
        for k, (i, j) in enumerate(pairs):
            for b in range(B if i < numVeh else 1):
                (ka, a), (kb, c) = obj(b, i), obj(b, j)
                if ka == 'poly' and kb == 'curve':
                    (ka, a), (kb, c) = (kb, c), (ka, a)
                groups.setdefault((ka, kb, a.shape, c.shape), []).append((b, k, a, c))
        for (ka, kb, _, _), items in groups.items():
            A = np.stack([it[2] for it in items])
            C = np.stack([it[3] for it in items])
            if ka == 'curve' and kb == 'curve':
                out, st = _bez.min_dist_batch(A, C, max_depth=self.spatial_max_depth,
                                              max_nodes=self.spatial_max_nodes)
            elif ka == 'curve':
                o5, st = _bez.min_dist2poly_batch(A, C, max_depth=self.spatial_max_depth,
                                                  max_nodes=self.spatial_max_nodes)
                # (alpha, t1, closest point) has no second curve parameter: the third column
                # repeats alpha (a duplicate of the distance constraint)
                out = np.stack([o5[:, 0], o5[:, 1], o5[:, 0]], axis=1)
                st = st & ~2                   # bit 2 only says "no closest point reported"
            else:
                from .gjk import gjk as _gjk
                flag, _, _, d = _gjk.gjk_batch(A, C)
                alpha = np.where(flag > 0, d, 0.0)
                out = np.stack([alpha, alpha, alpha], axis=1)
                st = np.where(flag < 0, 8, 0).astype(np.int32)
            for (b, k, _, _), o, s in zip(items, out, st):
                rows[b, k], status[b, k] = o, s
        for k, (i, j) in enumerate(pairs):
            if i >= numVeh:
                rows[1:, k], status[1:, k] = rows[0, k], status[0, k]
        return rows, status

    def _spatial_check(self, status):
        self.last_status = status
        bad = int((status != 0).sum())
        if bad and self.spatial_on_limit == 'raise':
            raise RecursionError('minDist exceeded its depth/node budget on %d of %d pairs (status codes '
                                 'in last_status); the reference recurses without bound on such pairs '
                                 '(SURVEY Q6). Set spatial_on_limit = "nan" to get NaN rows instead.'
                                 % (bad, status.size))

    def spatialSeparationConstraints(self, x):
        """optimization.py:109-133: all pairs among the vehicles and the shape
        obstacles, minDist - maxSep; like the reference the (alpha, t1, t2) tuple is
        kept, so the result is [npairs, 3] (SURVEY Q7).  One warp per pair, one launch
        per group of equally shaped pairs."""
        y = self.reshapeVector(x)
        rows, status = self._spatial_rows(y[None])
        self._spatial_check(status[0])
        return rows[0] - self.model['maxSep']

    @_on_model_device
    def spatialSeparationConstraints_jac(self, x):
        """Additive: the '2-point' FD Jacobian SLSQP would form from nvar+1 calls of
        spatialSeparationConstraints, [npairs*3, nvar]: the base point and all perturbed
        points go through the minDist kernel in ONE launch per pair group ((nvar+1) x pairs
        warps); obstacle-obstacle rows are constants (zero rows)."""
        x = np.asarray(x, dtype=np.float64)
        eng = self._engine(with_obstacles=False)
        Xp, d_dx = eng.fd_points(x)
        cpts, _ = eng.assemble(Xp.view(x.size + 1, x.size), 0)
        nrow = self.model['dim'] * (self.model['deg'] + 1)
        Y = eng.download(cpts[:, :, :nrow].contiguous(), key="spatial_y")
        Y = Y.reshape(x.size + 1, self.model['numVeh'] * self.model['dim'], self.model['deg'] + 1)
        rows, status = self._spatial_rows(Y)
        self._spatial_check(status)
        F = rows.reshape(x.size + 1, -1)
        dx = eng.download(d_dx)[0]
        return ((F[1:] - F[0]) / dx[:, None]).T

    @property
    def minSpeedConstraints(self):
        """optimization.py:135-151 -> _minSpeedConstraints (:349-384)."""
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            E = _deg_elev()
            cpts, tf = eng.assemble(eng.upload(x), E)
            out = eng.speed(cpts, tf, E, 1.0, -float(self.model['minSpeed']) ** 2)
            return eng.download(out, key="out:minspeed", copy=not self.zero_copy_results).reshape(-1)
        return wrapper

    @property
    def maxSpeedConstraints(self):
        """optimization.py:153-169 -> _maxSpeedConstraints (:387-422)."""
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            E = _deg_elev()
            cpts, tf = eng.assemble(eng.upload(x), E)
            out = eng.speed(cpts, tf, E, -1.0, float(self.model['maxSpeed']) ** 2)
            return eng.download(out, key="out:maxspeed", copy=not self.zero_copy_results).reshape(-1)
        return wrapper

    @property
    def maxAngularRateConstraints(self):
        """optimization.py:171-187 -> _maxAngularRateConstraints (:425-459)."""
        def wrapper(x):
            if self.model['dim'] != 2:                      # optimization.py:590-593
                msg = ('The input curve must be two dimensional,\n'
                       'instead it is {} dimensional'.format(self.model['dim']))
                raise ValueError(msg)
            eng = self._engine(with_obstacles=False)
            E = _deg_elev()
            cpts, tf = eng.assemble(eng.upload(x), E)
            out = eng.angrate(cpts, tf, E, -1.0, float(self.model['maxAngRate']) ** 2)
            return eng.download(out, key="out:angrate", copy=not self.zero_copy_results).reshape(-1)
        return wrapper

    # ------------------------------------------------------------------
    # additive: Jacobians of the closures above, J[m, nvar], equal to what SLSQP
    # would form by nvar+1 calls (SciPy's '2-point' rule and step), computed in one
    # batched launch.  Hand them to SciPy as {'type': 'ineq', 'fun': f, 'jac': f_jac}.
    @property
    def temporalSeparationConstraints_jac(self):
        def wrapper(x):
            eng = self._engine(with_obstacles=True)
            if eng.N <= 1:
                return None
            JT = eng.jac_separation(x, _deg_elev(), dense=True)
            return eng.download(JT, key="jac:sep", copy=not self.zero_copy_results).T
        return wrapper

    @property
    def maxSpeedConstraints_jac(self):
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            JT = eng.jac_speed(x, _deg_elev(), -1.0, dense=True)
            return eng.download(JT, key="jac:maxspeed", copy=not self.zero_copy_results).T
        return wrapper

    @property
    def minSpeedConstraints_jac(self):
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            JT = eng.jac_speed(x, _deg_elev(), 1.0, dense=True)
            return eng.download(JT, key="jac:minspeed", copy=not self.zero_copy_results).T
        return wrapper

    @property
    def maxAngularRateConstraints_jac(self):
        """Batched literal FD (no closed form for the ratio): same noise floor
        as SciPy differencing the reference (~1e-7 relative)."""
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            JT = eng.jac_angrate(x, _deg_elev(), -1.0, float(self.model['maxAngRate']) ** 2)
            return eng.download(JT, key="jac:angrate", copy=not self.zero_copy_results).T
        return wrapper

    @property
    def maxAngularRateConstraints_jac_closed(self):
        """The same quotient in closed form (ConstraintEngine.jac_angrate_closed): no perturbed
        points are evaluated, no differencing noise (agrees with the exactly rounded quotient to
        ~1e-9), and a control-point variable touches only its own vehicle's rows.  n + DEG_ELEV
        <= 127; the literal closure above covers larger degrees."""
        def wrapper(x):
            eng = self._engine(with_obstacles=False)
            JT = eng.jac_angrate_closed(x, _deg_elev(), -1.0)
            return eng.download(JT, key="jac:angrate_closed", copy=not self.zero_copy_results).T
        return wrapper

    # ------------------------------------------------------------------
    def generateGuess(self, std=0, seed=None):
        """Initial guess of optimization.py:189-240 (host logic): per vehicle the straight
        line between its end points -- for Dubins models between the second and the
        penultimate control point, which the end speeds and headings pin -- sampled at the
        free control points, plus N(0, std) noise.  numpy's global RNG is seeded and drawn
        from in the reference's order (vehicle-major, one draw of a full row per
        dimension), so seeded guesses are identical."""
        m = self.model
        deg, dim, tf = m['deg'], m['dim'], m['tf']
        dubins = m['initSpeeds'][0] is not None
        if dubins and dim != 2:
            raise ValueError('The dimension must be 2 for initial and final speeds and angles.')
        npts = deg - 1 if dubins else deg + 1
        np.random.seed(seed)
        rows = []
        for veh in range(m['numVeh']):
            first = [m['initPoints'][veh, axis] for axis in range(dim)]
            last = [m['finalPoints'][veh, axis] for axis in range(dim)]
            if dubins:
                lead_in = m['initSpeeds'][veh] * tf / deg
                lead_out = m['finalSpeeds'][veh] * tf / deg
                heading_in = (np.cos(m['initAngs'][veh]), np.sin(m['initAngs'][veh]))
                heading_out = (np.cos(m['finalAngs'][veh]), np.sin(m['finalAngs'][veh]))
                first = [first[axis] + lead_in * heading_in[axis] for axis in range(dim)]
                last = [last[axis] - lead_out * heading_out[axis] for axis in range(dim)]
            for axis in range(dim):
                row = np.linspace(first[axis], last[axis], npts)
                row += np.random.randn(npts) * std
                rows.append(row[1:-1])
        if m['minGoal'].lower() == 'timeopt':
            rows.append([tf])
        return np.concatenate(rows)

    @_on_model_device
    def reshapeVector(self, x):
        """optimization.py:242-285, evaluated by the device assemble kernel
        (the same one every constraint closure uses) and copied back as the
        reference's [numVeh*dim, deg+1] matrix."""
        eng = self._engine(with_obstacles=False)
        cpts, _ = eng.assemble(eng.upload(x), 0)             # [1, numVeh, S]
        rows = self.model['dim'] * (self.model['deg'] + 1)
        y = eng.download(cpts[0, :, :rows].contiguous())
        return y.reshape(self.model['numVeh'] * self.model['dim'], self.model['deg'] + 1)

    # ------------------------------------------------------------------
    # additive, batched API
    @_on_model_device
    def evaluate_batch(self, X, which=('sep', 'maxspeed'), elev=None):
        """Evaluates the named constraint blocks for every row of X [B, nvar]
        in one pass; returns device tensors {name: [B, m_name]}."""
        E = _deg_elev() if elev is None else int(elev)
        res = {}
        if 'sep' in which:
            eng = self._engine(with_obstacles=True)
            d_x = X if isinstance(X, torch.Tensor) else eng.upload(X)
            cpts, _ = eng.assemble(d_x, E)
            res['sep'] = eng.separation(cpts, E, self.model['maxSep']).reshape(d_x.shape[0], -1)
        eng = self._engine(with_obstacles=False)
        if 'maxspeed' in which or 'minspeed' in which:
            d_x = X if isinstance(X, torch.Tensor) else eng.upload(X)
            cpts, tf = eng.assemble(d_x, E)
            if 'maxspeed' in which:
                res['maxspeed'] = eng.speed(cpts, tf, E, -1.0, float(self.model['maxSpeed']) ** 2
                                            ).reshape(d_x.shape[0], -1)
            if 'minspeed' in which:
                res['minspeed'] = eng.speed(cpts, tf, E, 1.0, -float(self.model['minSpeed']) ** 2
                                            ).reshape(d_x.shape[0], -1)
        return res

    @_on_model_device
    def jacobian_batch(self, X, which=('sep', 'maxspeed'), elev=None):
        """The Jacobian counterpart of evaluate_batch: SciPy's 2-point J^T of the named blocks
        ('sep', 'maxspeed', 'minspeed') at every row of X [B, nvar] (host or device), in closed
        form and one launch per block; returns device tensors {name: J^T [B, nvar, m_name]}
        (row b equals the transposed result of the *_jac closure at X[b])."""
        E = _deg_elev() if elev is None else int(elev)
        res = {}
        if 'sep' in which:
            eng = self._engine(with_obstacles=True)
            if eng.N <= 1:
                B = int(X.shape[0]) if isinstance(X, torch.Tensor) else np.atleast_2d(X).shape[0]
                res['sep'] = torch.empty((B, eng.nvar, 0), dtype=torch.float64, device=eng.device)
            else:
                res['sep'] = eng.jac_separation(X, E, dense=True)
        if 'maxspeed' in which or 'minspeed' in which:
            eng = self._engine(with_obstacles=False)
            base = eng._fd_base(X, E)
            if 'maxspeed' in which:
                res['maxspeed'] = eng.jac_speed(None, E, -1.0, base=base)
            if 'minspeed' in which:
                res['minspeed'] = eng.jac_speed(None, E, 1.0, base=base)
        return res

    @_on_model_device
    def evaluate_reduced(self, X, elev=None):
        """Additive API for swarms whose full constraint vector is consumed on the
        device (508 MB per x at N=1024): host X [B, nvar] -> host arrays
        ``pairmin`` [B, P] (min over each pair's elevated separation values; its
        sign is the active-pair flag) and ``maxspeed`` [B, numVeh*L].  Every
        separation row is still materialised in HBM and stays available as the
        device tensor ``self.workspace['sep']`` until the next call."""
        E = _deg_elev() if elev is None else int(elev)
        eng = self._engine(with_obstacles=True)
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        B = X.shape[0]
        P = _engine.num_pairs(eng.N)
        L = 2 * self.model['deg'] + E + 1
        ws = getattr(self, 'workspace', None)
        if ws is None or ws.get('key') != (B, E):
            ws = {'key': (B, E),
                  'sep': torch.empty((B, P, L), dtype=torch.float64, device=eng.device),
                  'pairmin': torch.empty((B, P), dtype=torch.float64, device=eng.device),
                  'maxspeed': torch.empty((B, self.model['numVeh'], L), dtype=torch.float64,
                                          device=eng.device)}
            self.workspace = ws
        cpts, tf = eng.assemble(eng.upload(X), E)
        eng.separation(cpts, E, self.model['maxSep'], out=ws['sep'], pairmin=ws['pairmin'])
        eng.speed(cpts, tf, E, -1.0, float(self.model['maxSpeed']) ** 2, nveh=self.model['numVeh'],
                  out=ws['maxspeed'])
        # two async copies into pinned staging, one synchronisation
        pm = eng._pinned_buf('pairmin', ws['pairmin'].numel())
        sp = eng._pinned_buf('maxspeed', ws['maxspeed'].numel())
        pm.copy_(ws['pairmin'].view(-1), non_blocking=True)
        sp.copy_(ws['maxspeed'].view(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        pmh, sph = pm.numpy().reshape(B, P), sp.numpy().reshape(B, -1)
        if not self.zero_copy_results:
            pmh, sph = pmh.copy(), sph.copy()
        return {'pairmin': pmh, 'maxspeed': sph}

    @_on_model_device
    def evaluate_sweep(self, X, elev=None, chunk=4, out=None):
        """Pipelined form of :meth:`evaluate_reduced` for the nvar+1 points of a finite
        difference sweep (SciPy asks for them one by one, `_numdiff.py:683-712`; here the
        caller hands all of them over): host X [M, nvar] is processed in chunks of
        ``chunk`` rows with two device workspaces, so that the pinned host->device copy
        and the kernels of chunk k+1 overlap the device->host copy of chunk k (separate
        copy stream, events, no host synchronisation inside the loop).  Returns host
        arrays ``pairmin`` [M, P] and ``maxspeed`` [M, numVeh*L] (pinned; reused by the
        next call unless ``out`` supplies the destination dict of pinned tensors)."""
        E = _deg_elev() if elev is None else int(elev)
        eng = self._engine(with_obstacles=True)
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        M = X.shape[0]
        if X.shape[1] != eng.nvar:
            raise ValueError("x has %d entries, the model expects %d" % (X.shape[1], eng.nvar))
        P = _engine.num_pairs(eng.N)
        L = 2 * self.model['deg'] + E + 1
        nv = self.model['numVeh']
        chunk = max(1, min(int(chunk), M))
        sw = getattr(self, '_sweep_ws', None)
        if sw is None or sw['key'] != (chunk, E):
            def wsset():
                return {'x': torch.empty((chunk, eng.nvar), dtype=torch.float64, device=eng.device),
                        'sep': torch.empty((chunk, P, L), dtype=torch.float64, device=eng.device),
                        'pairmin': torch.empty((chunk, P), dtype=torch.float64, device=eng.device),
                        'maxspeed': torch.empty((chunk, nv, L), dtype=torch.float64, device=eng.device),
                        'done': None}
            sw = {'key': (chunk, E), 'sets': [wsset(), wsset()], 'copy_stream': torch.cuda.Stream(device=eng.device),
                  'copy_stream2': torch.cuda.Stream(device=eng.device),
                  'upload_stream': torch.cuda.Stream(device=eng.device)}
            self._sweep_ws = sw
        if out is None:
            out = {'pairmin': eng._pinned_buf('sweep_pairmin', M * P).view(M, P),
                   'maxspeed': eng._pinned_buf('sweep_maxspeed', M * nv * L).view(M, nv * L)}
        xs = eng._pinned_buf('sweep_x', X.size).view(M, eng.nvar)
        xs_np = xs.numpy()                           # filled chunk by chunk, just ahead of each upload
        main, side, side2 = torch.cuda.current_stream(), sw['copy_stream'], sw['copy_stream2']
        up = sw['upload_stream']
        max_speed2 = float(self.model['maxSpeed']) ** 2

        def upload(k, after):
            # x of chunk k goes up one step ahead on its own stream, so that it never queues
            # behind the result copies of the previous chunk on a shared copy engine
            lo_ = k * chunk
            hi_ = min(M, lo_ + chunk)
            xs_np[lo_:hi_] = X[lo_:hi_]
            with torch.cuda.stream(up):
                if after is not None:
                    up.wait_event(after)             # kernels that last read this set's x
                sw['sets'][k & 1]['x'][:hi_ - lo_].copy_(xs[lo_:hi_], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(up)
            return ev

        nchunks = (M + chunk - 1) // chunk
        up.wait_stream(main)
        x_ready = upload(0, None)
        prev_ready = None
        for k, lo in enumerate(range(0, M, chunk)):
            hi = min(M, lo + chunk)
            b = hi - lo
            ws = sw['sets'][k & 1]
            if ws['done'] is not None:
                main.wait_event(ws['done'])          # D2H of the chunk that used this set two steps ago
            main.wait_event(x_ready)
            if k + 1 < nchunks:
                x_ready = upload(k + 1, prev_ready)
            cpts, tf = eng.assemble(ws['x'][:b], E)
            # speed rows first (see evaluate_sweep_active.launch)
            eng.speed(cpts, tf, E, -1.0, max_speed2, nveh=nv, out=ws['maxspeed'][:b])
            eng.separation(cpts, E, self.model['maxSep'], out=ws['sep'][:b], pairmin=ws['pairmin'][:b])
            ready = torch.cuda.Event()
            ready.record(main)
            prev_ready = ready
            # the two result blocks leave on two copy streams (two copy engines share the link)
            with torch.cuda.stream(side2):
                side2.wait_event(ready)
                out['maxspeed'][lo:hi].copy_(ws['maxspeed'][:b].view(b, -1), non_blocking=True)
                done2 = torch.cuda.Event()
                done2.record(side2)
            with torch.cuda.stream(side):
                side.wait_event(ready)
                out['pairmin'][lo:hi].copy_(ws['pairmin'][:b], non_blocking=True)
                side.wait_event(done2)
                ws['done'] = torch.cuda.Event()
                ws['done'].record(side)
        side.synchronize()
        main.synchronize()
        self.workspace = {'key': None, 'sep': sw['sets'][(k & 1)]['sep']}
        return {'pairmin': out['pairmin'].numpy(), 'maxspeed': out['maxspeed'].numpy()}

    @_on_model_device
    def evaluate_sweep_active(self, X, elev=None, chunk=4, threshold=0.0, rows=True):
        """Like :meth:`evaluate_sweep`, but only the *reduced* result of every evaluation leaves
        the device: the packed active bitmask of all pairs (1 bit per pair: min over the pair's
        L values < ``threshold``), the compacted (pair, min) list of the active pairs, the
        per-vehicle minima of the max-speed block and their bitmask.  The fp64 [chunk, P]
        per-pair-minimum matrix, and with ``rows=True`` (default) every elevated row, are still
        produced in HBM for device-side consumers (``self.workspace``).  At N = 1024 that is
        ~0.4 MB per 4 evaluations over PCIe instead of 20.7 MB (per-pair minima + speed rows)
        or 2 GB (the full vectors).  Returns a :class:`SweepActive`.

        A chunk whose active list overflows its capacity (sized from the previous calls) is
        recomputed at the end with a larger list, so the result is always complete."""
        E = _deg_elev() if elev is None else int(elev)
        eng = self._engine(with_obstacles=True)
        X = np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))
        M = X.shape[0]
        if X.shape[1] != eng.nvar:
            raise ValueError("x has %d entries, the model expects %d" % (X.shape[1], eng.nvar))
        P = _engine.num_pairs(eng.N)
        L = 2 * self.model['deg'] + E + 1
        nv = self.model['numVeh']
        chunk = max(1, min(int(chunk), M))
        nchunks = (M + chunk - 1) // chunk
        sw = getattr(self, '_active_ws', None)
        cap = max(1024, int(getattr(self, '_active_cap', 0)), (chunk * P) // 32)
        if sw is None or sw['key'] != (chunk, E, bool(rows), cap, float(threshold), eng.dev_index):
            dev = eng.device

            def wsset():
                return {'x': torch.empty((chunk, eng.nvar), dtype=torch.float64, device=dev),
                        'sep': torch.empty((chunk, P, L), dtype=torch.float64, device=dev) if rows else None,
                        'pairmin': torch.empty((chunk, P), dtype=torch.float64, device=dev),
                        'maxspeed': torch.empty((chunk, nv, L), dtype=torch.float64, device=dev),
                        'vehmin': torch.empty((chunk, nv), dtype=torch.float64, device=dev),
                        'pairs': _engine.ActiveSet(chunk * P, cap, dev, threshold),
                        'vehs': _engine.ActiveSet(chunk * nv, 0, dev, 0.0),
                        'done': None}
            sw = {'key': (chunk, E, bool(rows), cap, float(threshold), eng.dev_index), 'sets': [wsset(), wsset()],
                  'copy_stream': torch.cuda.Stream(device=dev), 'upload_stream': torch.cuda.Stream(device=dev)}
            self._active_ws = sw
        pslots, vslots = sw['sets'][0]['pairs'].nslots, sw['sets'][0]['vehs'].nslots
        out_pairs = eng._pinned_buf_i64('active_pairs', nchunks * pslots).view(nchunks, pslots)
        out_vehs = eng._pinned_buf_i64('active_vehs', nchunks * vslots).view(nchunks, vslots)
        out_vmin = eng._pinned_buf('active_vehmin', M * nv).view(M, nv)
        xs = eng._pinned_buf('sweep_x', X.size).view(M, eng.nvar)
        xs_np = xs.numpy()
        with torch.cuda.device(eng.device):
            main, side, up = torch.cuda.current_stream(), sw['copy_stream'], sw['upload_stream']
            max_speed2 = float(self.model['maxSpeed']) ** 2

            def upload(k, after):
                lo_ = k * chunk
                hi_ = min(M, lo_ + chunk)
                xs_np[lo_:hi_] = X[lo_:hi_]
                with torch.cuda.stream(up):
                    if after is not None:
                        up.wait_event(after)
                    sw['sets'][k & 1]['x'][:hi_ - lo_].copy_(xs[lo_:hi_], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(up)
                return ev

            def launch(ws, b, pa, va):
                # the speed rows go first: behind the persistent pair kernel they would find no SM until the NEXT
                # chunk's pair kernel (already queued on the other stream) has drained, and this chunk's result
                # would leave the device a whole kernel late
                pa.reset()
                cpts, tf = eng.assemble(ws['x'][:b], E)
                eng.speed(cpts, tf, E, -1.0, max_speed2, nveh=nv, out=ws['maxspeed'][:b], vehmin=ws['vehmin'][:b],
                          active=va)
                eng.separation(cpts, E, self.model['maxSep'], out=ws['sep'][:b] if rows else None, rows=rows,
                               pairmin=ws['pairmin'][:b], active=pa)

            use_graph = bool(getattr(self, 'sweep_cuda_graphs', True))
            # Consecutive chunks run on two alternating compute streams (their workspaces are
            # disjoint): the next chunk's kernels are already queued when the persistent pair kernel
            # of the current one drains, so its CTAs fill the SMs as they free up -- no launch gap and
            # no idle tail between chunks.
            lanes = sw.setdefault('compute_streams', [torch.cuda.Stream(device=eng.device) for _ in range(2)])
            for st in lanes:
                st.wait_stream(main)
            up.wait_stream(main)
            x_ready = upload(0, None)
            prev_ready = None
            for k, lo in enumerate(range(0, M, chunk)):
                hi = min(M, lo + chunk)
                b = hi - lo
                ws = sw['sets'][k & 1]
                st = lanes[k & 1]
                with torch.cuda.stream(st):
                    if ws['done'] is not None:
                        st.wait_event(ws['done'])
                    st.wait_event(x_ready)
                    if k + 1 < nchunks:
                        x_ready = upload(k + 1, prev_ready)
                    if b != chunk:                          # ragged last chunk: its own, smaller destinations
                        pa = _engine.ActiveSet(b * P, cap, eng.device, threshold)
                        va = _engine.ActiveSet(b * nv, 0, eng.device, 0.0)
                        launch(ws, b, pa, va)
                    else:
                        pa, va = ws['pairs'], ws['vehs']
                        if ws.get('graph') is None and use_graph:
                            # the fixed launch sequence of a full chunk (counter reset, assemble, fused
                            # pair kernel, speed kernel) replays as one CUDA graph: no launch gaps
                            launch(ws, b, pa, va)                   # warm-up: plans, kernel attributes
                            st.synchronize()
                            ws['graph'] = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(ws['graph']):
                                launch(ws, b, pa, va)
                        if ws.get('graph') is not None:
                            ws['graph'].replay()
                        else:
                            launch(ws, b, pa, va)
                    ready = torch.cuda.Event()
                    ready.record(st)
                prev_ready = ready
                with torch.cuda.stream(side):
                    side.wait_event(ready)
                    out_pairs[k, :pa.nslots].copy_(pa.buf, non_blocking=True)
                    out_vehs[k, :va.nslots].copy_(va.buf, non_blocking=True)
                    out_vmin[lo:hi].copy_(ws['vehmin'][:b], non_blocking=True)
                    ws['done'] = torch.cuda.Event()
                    ws['done'].record(side)
            for st in lanes:
                main.wait_stream(st)
            side.synchronize()
            main.synchronize()
            res = SweepActive(out_pairs.numpy(), out_vehs.numpy(), out_vmin.numpy(), M, chunk, P, nv, cap)
            # overflowing lists: recompute those chunks (minima only) with a list that holds every pair
            worst = int(res.pair_counts().max()) if nchunks else 0
            for k in np.nonzero(res.pair_counts() > cap)[0]:
                lo, hi = k * chunk, min(M, k * chunk + chunk)
                big = _engine.ActiveSet((hi - lo) * P, (hi - lo) * P, eng.device, threshold)
                cpts, _ = eng.assemble(eng.upload(X[lo:hi]), E)
                pm = torch.empty((hi - lo, P), dtype=torch.float64, device=eng.device)
                eng.separation(cpts, E, self.model['maxSep'], rows=False, pairmin=pm, active=big)
                stage = eng._pinned_buf_i64("active_override", big.nslots)
                stage.copy_(big.buf, non_blocking=True)
                main.synchronize()
                res.overrides[int(k)] = stage.numpy().copy()
            self._active_cap = max(int(getattr(self, '_active_cap', 0)), int(1.25 * worst) + 64)
            self.workspace = {'key': None, 'sep': sw['sets'][(nchunks - 1) & 1]['sep'],
                              'pairmin': sw['sets'][(nchunks - 1) & 1]['pairmin']}
        return res

    # -- cost callables (A14, optimization.py:287-308) -----------------------
    @_on_model_device
    def _objective(self, x, kind):
        """One launch for every row of x: a 1-D x gives a float (the reference's
        callable), a 2-D batch [B, nvar] gives float64[B]."""
        eng = self._engine(with_obstacles=False)
        E = _deg_elev()
        single = np.ndim(x) == 1
        d_x = eng.upload(x)
        cpts, tf = eng.assemble(d_x, E)
        out = torch.empty((d_x.shape[0],), dtype=torch.float64, device=eng.device)
        plan = eng.plan(E)
        if kind == 'euclidean':
            _engine._capi.call("bez_objective_euclidean", plan.handle, _engine._ptr(cpts), int(d_x.shape[0]),
                               eng.N, eng.numVeh, _engine._ptr(out), eng._st())
        else:
            # the reference passes model['tf'] here even for time-optimal problems
            tfm = torch.full_like(tf, float(self.model['tf']))
            _engine._capi.call("bez_objective_accel", plan.handle, _engine._ptr(cpts), _engine._ptr(tfm),
                               int(d_x.shape[0]), eng.N, eng.numVeh, _engine._ptr(out), eng._st())
        host = eng.download(out, key="out:objective")
        return float(host[0]) if single else host

    @_on_model_device
    def _objective_grad(self, x, kind):
        """SciPy's '2-point' gradient of the objective (what SLSQP forms with nvar+1 calls,
        _slsqp_py.py:424-426) in one launch, cancellation free (bez_objective_grad)."""
        eng = self._engine(with_obstacles=False)
        E = _deg_elev()
        x = np.asarray(x, dtype=np.float64)
        _, dx = eng.fd_steps(x)
        nvarN = eng.numVeh * eng.dim * eng.ncols
        grad = np.zeros(x.size)
        if nvarN:
            cpts, _ = eng.assemble(eng.upload(x), E)
            d_dx = torch.as_tensor(dx[:nvarN], device=eng.device)
            out = torch.empty((nvarN,), dtype=torch.float64, device=eng.device)
            _engine._capi.call("bez_objective_grad", eng.plan(E).handle, _engine._ptr(cpts),
                               0 if kind == 'euclidean' else 1, float(self.model['tf']), eng.numVeh, eng.ncols,
                               eng.offset, _engine._ptr(d_dx), _engine._ptr(out), eng._st())
            grad[:nvarN] = eng.download(out, key="out:objective_grad")
        # a tf variable (time-optimal models) does not enter these two objectives: the
        # reference evaluates them with model['tf'] and the end-speed control points of a
        # Dubins model follow x[-1], which Euclidean/Accel models do not have
        return grad

    @property
    def objectiveFunction_jac(self):
        """Additive: gradient of :attr:`objectiveFunction` for ``minimize(jac=...)``, equal to
        SciPy's own 2-point finite difference of the callable (exactly rounded quotient)."""
        minGoal = self.model['minGoal'].lower()
        if minGoal == 'euclidean':
            return lambda x: self._objective_grad(x, 'euclidean')
        if minGoal == 'accel':
            return lambda x: self._objective_grad(x, 'accel')
        if minGoal == 'timeopt':
            def grad(x):                 # ((x[-1] + h) - x[-1]) / dx = 1 exactly
                g = np.zeros(np.size(x))
                g[-1] = 1.0
                return g
            return grad
        self.objectiveFunction          # raises the reference's ValueError for unknown goals
        raise NotImplementedError("no gradient for the %r objective" % minGoal)

    def euclideanObjective(self, x):
        """optimization.py:287-292 -> _euclideanObjective (:462-489)"""
        return self._objective(x, 'euclidean')

    def accelObjective(self, x):
        """optimization.py:294-300 -> _minAccelObjective (:503-519)"""
        return self._objective(x, 'accel')

    def jerkObjective(self, x):
        """optimization.py:302-308: the reference's _minJerkObjective is an @njit
        over Python objects and raises a numba TypingError when called (SURVEY Q10)."""
        raise NotImplementedError("the reference's jerk objective cannot run (numba TypingError); not provided")
