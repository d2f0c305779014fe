"""Closed-form angular-rate Jacobian (bez_jac_angrate_sq, ConstraintEngine.jac_angrate_closed,
BezOptimization.maxAngularRateConstraints_jac_closed, ProblemBatch "angrate_closed").
Judged like the separation and speed blocks: block-relative 1e-9 against the exactly rounded
2-point quotient of the oracle (rational arithmetic on the fp64 points)."""
import ctypes

import numpy as np
import pytest

from conftest import relerr

JTOL = 1e-9


@pytest.fixture(scope="module")
def gopt():
    import torch
    assert torch.cuda.is_available()
    from optimalbeziertrajectorygeneration_b200 import optimization
    yield optimization
    optimization.DEG_ELEV = 0


EX1 = dict(numVeh=2, dimension=2, degree=10, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=5,
           maxAngRate=1, initPoints=[(0, 5), (3, 0)], finalPoints=[(8, 4), (7, 10)],
           initSpeeds=[1, 1], finalSpeeds=[1, 1], initAngs=[0, np.pi / 2],
           finalAngs=[0, np.pi / 2], pointObstacles=[[3, 2], [6, 7]])


def _exact(args, x, E, cols=None):
    """Exactly rounded SciPy quotient of the angular-rate block, columns ``cols`` (default all)."""
    from oracle import bezier_oracle as O
    fun = O.make_callables(O.Model(**args), E, dtype=object)["angrate"]
    x = np.asarray(x, dtype=np.float64)
    cols = range(x.size) if cols is None else cols
    h, dx = O.fd_steps(x)
    f0 = fun(O._cast(x, object))
    J = np.empty((f0.size, len(cols)))
    for i, k in enumerate(cols):
        x1 = x.copy()
        x1[k] = x[k] + h[k]
        q = (fun(O._cast(x1, object)) - f0) / O._num(float(dx[k]), object)
        J[:, i] = [float(v) for v in q]
    return J


def _check_exact(gopt, args, x, E, cols=None):
    b = gopt.BezOptimization(**args)
    gopt.DEG_ELEV = E
    J = b.maxAngularRateConstraints_jac_closed(x)
    assert J.shape == (b.model['numVeh'] * (4 * (b.model['deg'] + E) + 1), b.nvar)
    if cols is not None:
        J = J[:, cols]
    Jex = _exact(args, x, E, cols)
    scale = np.abs(Jex).max()
    assert np.abs(J - Jex).max() / scale < JTOL
    # rows of vehicles a variable does not move are exact zeros in both
    assert np.all(np.abs(Jex[J == 0]) <= 1e-13 * scale)
    assert np.all(np.abs(J[Jex == 0]) <= 1e-13 * scale)
    return J


def _c5():
    from oracle.make_golden import dubins_problem_args
    return dubins_problem_args(0)


@pytest.mark.gpu
@pytest.mark.parametrize("E", [0, 8, 30])
def test_exact_c5(gopt, golden, E):
    _check_exact(gopt, _c5(), golden("constraints")["c5_s0_x"], E)


@pytest.mark.gpu
def test_exact_c5_e100_columns(gopt, golden):
    """m = 110 (U1 = 14, the C5 shape): control points 0, 6, 13 and tf"""
    _check_exact(gopt, _c5(), golden("constraints")["c5_s0_x"], 100, cols=[0, 6, 13, 14])


@pytest.mark.gpu
@pytest.mark.parametrize("E", [0, 10])
def test_exact_example1(gopt, golden, E):
    _check_exact(gopt, EX1, golden("jacobian")["ex1_x"], E)


def _fixed_end(N, deg, goal, seed, tf=3.0):
    rng = np.random.default_rng(seed)
    args = dict(numVeh=N, dimension=2, degree=deg, minimizeGoal=goal, maxSep=0.5, maxAngRate=2.0, tf=tf,
                initPoints=rng.uniform(-5, 5, size=(N, 2)), finalPoints=rng.uniform(-5, 5, size=(N, 2)))
    nvar = N * 2 * (deg - 1) + (1 if goal == 'TimeOpt' else 0)
    x = rng.normal(size=nvar) * 2
    if goal == 'TimeOpt':
        x[-1] = 2.5
    return args, x


@pytest.mark.gpu
def test_exact_euclidean_three_vehicles(gopt):
    args, x = _fixed_end(3, 5, 'Euclidean', 1)
    _check_exact(gopt, args, x, 6)


@pytest.mark.gpu
def test_exact_timeopt_without_direction_rows(gopt):
    """tf scales the derivatives but moves no control point"""
    args, x = _fixed_end(2, 6, 'TimeOpt', 2)
    J = _check_exact(gopt, args, x, 4)
    assert np.abs(J[:, -1]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("deg,E,cols", [(5, 2, None), (6, 2, None), (7, 120, [0, 3, 11])])
def test_exact_block_edges(gopt, deg, E, cols):
    """m = 7 and 8 (one and two 8-blocks), m = 127 (the largest tensor-path shape)"""
    args, x = _fixed_end(1, deg, 'TimeOpt', 3)
    if cols is not None:
        cols = cols + [x.size - 1]
    _check_exact(gopt, args, x, E, cols)


@pytest.mark.gpu
def test_matches_literal_and_reference(gopt, golden):
    from oracle.make_golden import dubins_problem_args
    g = golden("jacobian")
    b = gopt.BezOptimization(**dubins_problem_args(5, nobs=4, deg=6))
    gopt.DEG_ELEV = 8
    J = b.maxAngularRateConstraints_jac_closed(g["dub_x"])
    assert relerr(J, b.maxAngularRateConstraints_jac(g["dub_x"])) < 1e-5
    assert relerr(J, g["dub_J_angrate_E8"]) < 1e-5


@pytest.mark.gpu
def test_layouts_and_batching(gopt, golden):
    import torch
    b = gopt.BezOptimization(**EX1)
    eng = b._engine(False)
    E = 10
    x = golden("jacobian")["ex1_x"]
    L4 = 4 * (10 + E) + 1
    JT = eng.jac_angrate_closed(x, E, -1.0).cpu().numpy()                     # [nvar, 2 L4]
    sw = eng.jac_angrate_closed(x, E, -1.0, dense=False).cpu().numpy()        # [2*2*ncols + 2, L4]
    nvarN = eng.numVeh * 2 * eng.ncols
    assert sw.shape == (nvarN + eng.numVeh, L4)
    for k in range(nvarN):
        v = k // (2 * eng.ncols)
        assert np.array_equal(sw[k], JT[k, v * L4:(v + 1) * L4])
        assert not np.any(JT[k, (1 - v) * L4:(2 - v) * L4])                   # the other vehicle's rows
    for v in range(eng.numVeh):
        assert np.array_equal(sw[nvarN + v], JT[-1, v * L4:(v + 1) * L4])
    X = np.stack([x, x + 0.01, x - 0.02])
    JB = eng.jac_angrate_closed(X, E, -1.0).cpu().numpy()
    for i in range(3):
        assert np.array_equal(JB[i], eng.jac_angrate_closed(X[i], E, -1.0).cpu().numpy())
    JD = eng.jac_angrate_closed(torch.as_tensor(X, device=eng.device), E, -1.0).cpu().numpy()
    assert np.array_equal(JD, JB)
    swB = eng.jac_angrate_closed(X, E, -1.0, dense=False).cpu().numpy()
    assert np.array_equal(swB[0], sw)


@pytest.mark.gpu
def test_problem_batch(gopt, golden):
    from oracle.make_golden import dubins_problem_args
    from optimalbeziertrajectorygeneration_b200.batch import ProblemBatch
    g = golden("constraints")
    seeds = (2, 0, 1, 0)
    sets = np.array([dubins_problem_args(s)["pointObstacles"] for s in seeds])
    template = {k: v for k, v in dubins_problem_args(seeds[0]).items() if k != "pointObstacles"}
    pb = ProblemBatch(template, sets)
    X = np.stack([g["c5_s%d_x" % s] for s in seeds])
    X[3] = X[3] + 0.01
    gopt.DEG_ELEV = 100
    out = pb.sweep(X, elev=100, blocks=("angrate_closed",))
    assert list(out) == ["angrate_closed"]
    f0, JT = out["angrate_closed"]
    assert tuple(JT.shape) == (4, pb.nvar, 441)
    for i, s in enumerate(seeds):
        b = gopt.BezOptimization(**dubins_problem_args(s))
        assert np.array_equal(f0[i].cpu().numpy(), b.maxAngularRateConstraints(X[i]))
        assert np.array_equal(JT[i].cpu().numpy().T, b.maxAngularRateConstraints_jac_closed(X[i]))


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_example1_slsqp_closed_jacobian(gopt):
    import scipy.optimize as sop
    gopt.DEG_ELEV = 0
    args = dict(EX1)
    bezopt = gopt.BezOptimization(**args)
    del args['pointObstacles']
    veh_only = gopt.BezOptimization(**args)
    x0 = bezopt.generateGuess(std=0)
    cons = [{'type': 'ineq', 'fun': veh_only.temporalSeparationConstraints,
             'jac': veh_only.temporalSeparationConstraints_jac},
            {'type': 'ineq', 'fun': bezopt.maxSpeedConstraints, 'jac': bezopt.maxSpeedConstraints_jac},
            {'type': 'ineq', 'fun': bezopt.maxAngularRateConstraints},
            {'type': 'ineq', 'fun': lambda x: x[-1]}]
    cons[2]['jac'] = bezopt.maxAngularRateConstraints_jac_closed
    res = sop.minimize(bezopt.objectiveFunction, x0=x0, method='SLSQP', constraints=cons,
                       jac=bezopt.objectiveFunction_jac, options={'maxiter': 250, 'disp': False})
    assert res.success
    assert res.fun == pytest.approx(2.4276431891903045, rel=2e-5)
    assert veh_only.temporalSeparationConstraints(res.x).min() > -1e-6
    assert bezopt.maxSpeedConstraints(res.x).min() > -1e-6
    assert bezopt.maxAngularRateConstraints(res.x).min() > -1e-6


@pytest.mark.gpu
def test_rejects_3d(gopt):
    from oracle.make_golden import synthetic_swarm_args
    args, x = synthetic_swarm_args(3)
    with pytest.raises(ValueError):
        gopt.BezOptimization(**args).maxAngularRateConstraints_jac_closed(x)


@pytest.mark.gpu
def test_degree_above_tensor_path(gopt):
    """n + E > 127: a clear error from the closed form; the literal closure still covers it"""
    from optimalbeziertrajectorygeneration_b200 import _capi
    args, x = _fixed_end(1, 8, 'TimeOpt', 4)
    b = gopt.BezOptimization(**args)
    gopt.DEG_ELEV = 120                                          # m = 128
    with pytest.raises(_capi.BezGpuError, match="127"):
        b.maxAngularRateConstraints_jac_closed(x)
    J = b.maxAngularRateConstraints_jac(x)
    assert J.shape == (4 * 128 + 1, b.nvar) and np.all(np.isfinite(J))


# ---- CPU: argument validation happens before any CUDA call ---------------------------------

class _FakeTables(ctypes.Structure):
    """Leading fields of bez_angrate_tables: the entry point reads n and m while validating."""
    _fields_ = [("n", ctypes.c_int), ("elev", ctypes.c_int), ("m", ctypes.c_int), ("device", ctypes.c_int),
                ("ptrs", ctypes.c_void_p * 5)]


def _lib():
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "optimalbeziertrajectorygeneration_b200", "libbezgpu.so")):
        sys.path.insert(0, root)
        import __graft_entry__ as g
        g.build()
    from optimalbeziertrajectorygeneration_b200 import _capi
    return _capi


def test_scratch_doubles_without_gpu():
    _capi = _lib()
    f = _capi.lib.bez_jac_angrate_scratch_doubles
    assert f(3, 2, 10, 100) == 3 * 2 * (128 * 14 + 432)          # m = 110: U = 14
    assert f(1, 1, 5, 2) == 128 * 1 + 432                        # m = 7: U = 1
    assert f(1, 1, 6, 2) == 128 * 2 + 432                        # m = 8: U = 2
    assert f(1, 1, 10, 118) == 0                                 # m = 128: unsupported


def test_argument_errors_without_gpu():
    _capi = _lib()
    fn = _capi.lib.bez_jac_angrate_sq
    buf = (ctypes.c_double * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    tabs = _FakeTables(10, 100, 110, 0)
    # Example1's shape: 2 vehicles, 7 free columns, tf
    good = dict(B=1, N=2, S=22, numVeh=2, ncols=7, offset=2, nvar=29, kdir=28, dense=1, ld=2 * 441)

    def call(tables, **kw):
        a = dict(good, **kw)
        return fn(tables, p, p, a["B"], a["N"], a["S"], a["numVeh"], a["ncols"], a["offset"], a["nvar"], p,
                  None, a["kdir"], -1.0, a["dense"], p, p, a["ld"], None)

    assert call(None) < 0
    assert "NULL" in _capi.last_error()
    assert call(ctypes.byref(tabs), nvar=30, kdir=29) < 0       # one variable too many
    assert "nvar" in _capi.last_error()
    assert call(ctypes.byref(tabs), kdir=3) < 0
    assert call(ctypes.byref(tabs), ld=441) < 0
    assert call(ctypes.byref(tabs), offset=6) < 0                # columns beyond control point n
    assert call(ctypes.byref(tabs), numVeh=3) < 0
    assert call(ctypes.byref(tabs), S=20) < 0
    big = _FakeTables(10, 118, 128, 0)
    assert call(ctypes.byref(big), ld=2 * 513) == -3             # BEZ_EUNSUPPORTED
    assert "127" in _capi.last_error()
