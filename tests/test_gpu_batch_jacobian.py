"""Batched closed-form separation and speed Jacobians (bez_jac_sepsq_elev_batched,
bez_jac_speed_sq_elev_batched, ConstraintEngine.jac_separation / jac_speed with x [B, nvar],
ProblemBatch "sep_closed" / "maxspeed_closed" / "minspeed_closed", BezOptimization.jacobian_batch).
Judged like the single-point blocks: block-relative 1e-9 against the exactly rounded 2-point
quotient of the oracle, and equal to the single-point closures problem by problem."""
import ctypes

import numpy as np
import pytest

JTOL = 1e-9
BLOCKS = ("sep", "maxspeed", "minspeed")


@pytest.fixture(scope="module")
def gopt():
    import torch
    assert torch.cuda.is_available()
    from optimalbeziertrajectorygeneration_b200 import optimization
    yield optimization
    optimization.DEG_ELEV = 0


@pytest.fixture(scope="module")
def batch_mod(gopt):
    from optimalbeziertrajectorygeneration_b200 import batch
    return batch


EX1 = dict(numVeh=2, dimension=2, degree=10, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=5,
           maxAngRate=1, initPoints=[(0, 5), (3, 0)], finalPoints=[(8, 4), (7, 10)],
           initSpeeds=[1, 1], finalSpeeds=[1, 1], initAngs=[0, np.pi / 2],
           finalAngs=[0, np.pi / 2], tf=10)


def _template(args):
    return {k: v for k, v in args.items() if k != "pointObstacles"}


def _fixed_end(V, dim, deg, goal, seed):
    rng = np.random.default_rng(seed)
    args = dict(numVeh=V, dimension=dim, degree=deg, minimizeGoal=goal, maxSep=0.8, maxSpeed=4.0, minSpeed=0.5,
                tf=12.0, initPoints=rng.uniform(-5, 5, size=(V, dim)), finalPoints=rng.uniform(-5, 5, size=(V, dim)))
    return args, rng


def _check_exact(J, Jex, what):
    assert J.shape == Jex.shape, what
    scale = np.abs(Jex).max()
    assert np.abs(J - Jex).max() / scale < JTOL, what
    # rows that do not depend on x_k are exact zeros in both (entries zero only by cancellation
    # may be O(ulp) instead of 0), as in the single-point checks
    assert np.all(np.abs(Jex[J == 0]) <= 1e-13 * scale), what
    assert np.all(np.abs(J[Jex == 0]) <= 1e-13 * scale), what


def _exact(args, x, E, name):
    from oracle import bezier_oracle as O
    fun = O.make_callables(O.Model(**args), E, dtype=object)[name]
    return O.fd_jacobian_exact(fun, x)


def _dubins_batch(M, nobs, deg, seed0=0):
    from oracle.make_golden import dubins_problem_args
    probs = [dubins_problem_args(seed0 + s, nobs=nobs, deg=deg) for s in range(M)]
    sets = np.stack([np.asarray(p["pointObstacles"], dtype=np.float64) for p in probs])
    return probs, sets


def _dubins_x(gopt, probs, seed):
    rng = np.random.default_rng(seed)
    g = gopt.BezOptimization(**probs[0]).generateGuess(std=0)
    X = g[None] + 0.3 * rng.standard_normal((len(probs), g.size))
    X[:, -1] = np.abs(X[:, -1]) + 4.0
    return X


# ---- 1. exact oracle ---------------------------------------------------------------------

@pytest.mark.gpu
def test_exact_problem_batch(gopt, batch_mod):
    """M = 3 Dubins problems with different obstacles, E = 8, through ProblemBatch.sweep"""
    E = 8
    probs, sets = _dubins_batch(3, nobs=4, deg=6)
    pb = batch_mod.ProblemBatch(_template(probs[0]), sets)
    X = _dubins_x(gopt, probs, 1)
    res = pb.sweep(X, elev=E, blocks=("sep_closed", "maxspeed_closed", "minspeed_closed"))
    L = 2 * 6 + E + 1
    for i, args in enumerate(probs):
        for name in BLOCKS:
            J = res[name + "_closed"][1][i].cpu().numpy().T
            Jex = _exact(args, X[i], E, name)
            if name == "sep":
                Jex = Jex[:pb.npairs_x * L]
            _check_exact(J, Jex, (i, name))


@pytest.mark.gpu
def test_exact_euclidean_3d(gopt):
    """fixed-end Euclidean 3-D model, several vehicles, B = 2 points through jacobian_batch"""
    E = 8
    args, rng = _fixed_end(3, 3, 5, 'Euclidean', 5)
    b = gopt.BezOptimization(**args)
    X = rng.normal(size=(2, b.nvar)) * 3
    res = b.jacobian_batch(X, which=BLOCKS, elev=E)
    for i in range(2):
        for name in BLOCKS:
            _check_exact(res[name][i].cpu().numpy().T, _exact(args, X[i], E, name), (i, name))


# ---- 2. batch equals single --------------------------------------------------------------

def _single(gopt, args, x, E):
    b = gopt.BezOptimization(**args)
    gopt.DEG_ELEV = E
    return {"sep": b.temporalSeparationConstraints_jac(x), "maxspeed": b.maxSpeedConstraints_jac(x),
            "minspeed": b.minSpeedConstraints_jac(x)}


@pytest.mark.gpu
@pytest.mark.parametrize("E", [0, 10])
def test_problem_batch_equals_single_example1(gopt, batch_mod, E):
    """Example1's 2-vehicle, 2-obstacle model with per-problem obstacles: the dense kernel on both
    sides, so the results are identical"""
    rng = np.random.default_rng(3)
    sets = rng.uniform(1.0, 9.0, size=(3, 2, 2))
    pb = batch_mod.ProblemBatch(EX1, sets)
    g = gopt.BezOptimization(**EX1).generateGuess(std=0)
    X = g[None] + 0.2 * rng.standard_normal((3, g.size))
    res = pb.sweep(X, elev=E, blocks=("sep_closed", "maxspeed_closed", "minspeed_closed"))
    L = 2 * 10 + E + 1
    for i in range(3):
        single = _single(gopt, dict(EX1, pointObstacles=[list(o) for o in sets[i]]), X[i], E)
        for name in BLOCKS:
            J = res[name + "_closed"][1][i].cpu().numpy().T
            Js = single[name][:pb.npairs_x * L] if name == "sep" else single[name]
            assert np.array_equal(J, Js), (i, name)


@pytest.mark.gpu
def test_problem_batch_equals_single_c5(gopt, batch_mod):
    """the C5 shape (n = 10, 16 obstacles, E = 100): batch and single-point closure both run the
    one-vehicle dense block as a tensor-path sweep, so the results are identical"""
    E = 100
    probs, sets = _dubins_batch(3, nobs=16, deg=10, seed0=20)
    pb = batch_mod.ProblemBatch(_template(probs[0]), sets)
    X = _dubins_x(gopt, probs, 2)
    res = pb.sweep(X, elev=E, blocks=("sep_closed", "maxspeed_closed", "minspeed_closed"))
    L = 2 * 10 + E + 1
    for i in range(3):
        single = _single(gopt, probs[i], X[i], E)
        for name in BLOCKS:
            J = res[name + "_closed"][1][i].cpu().numpy().T
            Js = single[name][:pb.npairs_x * L] if name == "sep" else single[name]
            assert np.array_equal(J, Js), (i, name)


@pytest.mark.gpu
def test_multi_start_points_equal_single_points(gopt):
    """B = 5 different x of one swarm model without obstacles (3-D Euclidean; 2-D TimeOpt with the
    angular-rate block): jac_*(X[i]) == jac_*(X)[i] bit for bit, both layouts, host and device input.
    TimeOpt without Dubins ends: tf moves no control point (no direction rows, zero separation tf rows)"""
    import torch
    E = 4
    for goal, dim in (("Euclidean", 3), ("TimeOpt", 2)):
        args, rng = _fixed_end(4, dim, 5, goal, 9)
        b = gopt.BezOptimization(**args)
        eng = b._engine(True)
        X = rng.normal(size=(5, b.nvar)) * 3
        if goal == "TimeOpt":
            X[:, -1] = np.abs(X[:, -1]) + 8.0
        jacs = {"sep": lambda x, dense: eng.jac_separation(x, E, dense=dense),
                "speed": lambda x, dense: eng.jac_speed(x, E, -1.0, dense=dense)}
        if dim == 2:
            jacs["angrate"] = lambda x, dense: eng.jac_angrate_closed(x, E, -1.0, dense=dense)
        d_X = torch.as_tensor(X, device=eng.device)
        for name, jac in jacs.items():
            for dense in (True, False):
                what = (goal, name, dense)
                JB = jac(X, dense).cpu().numpy()
                assert JB.shape[0] == 5, what
                assert np.array_equal(jac(d_X, dense).cpu().numpy(), JB), what
                for i in range(5):
                    assert np.array_equal(jac(X[i], dense).cpu().numpy(), JB[i]), what + (i,)
                    assert np.array_equal(jac(d_X[i], dense).cpu().numpy(), JB[i]), what + (i,)


# ---- 3. layouts --------------------------------------------------------------------------

def _sweep_to_dense_sep(sw, B, nvarN, N, numVeh, dim, ncols, L, npairs, kdir):
    """scatter the sweep layout [B][nvarN*(N-1) + ndir][L] into J^T [B][nvar][npairs*L]"""
    nvar = nvarN + (1 if kdir >= 0 else 0)
    out = np.zeros((B, nvar, npairs * L))
    v_of = np.arange(nvarN) // (dim * ncols)
    for k in range(nvarN):
        v = v_of[k]
        others = [u for u in range(N) if u != v]
        for uu, u in enumerate(others):
            i, j = min(v, u), max(v, u)
            p = i * (2 * N - i - 1) // 2 + (j - i - 1)
            out[:, k, p * L:(p + 1) * L] = sw[:, k * (N - 1) + uu]
    if kdir >= 0:
        out[:, kdir] = sw[:, nvarN * (N - 1):].reshape(B, npairs * L)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("V,dim,deg,E,B", [(9, 3, 10, 100, 3), (3, 2, 6, 60, 2), (4, 3, 5, 2, 3)])
def test_batched_sweep_rows_equal_dense_rows(gopt, V, dim, deg, E, B):
    """several vehicles: dense J^T on the dense kernel, the sweep layout on the tensor path where
    65 <= L <= 128 (V = 9, 3-D, n = 10, E = 100 runs the warp-specialised kernel: 1944 items per
    point, so tiles straddle variables, and the last tile of every point is partial)"""
    args, rng = _fixed_end(V, dim, deg, 'Euclidean', 11 + V)
    b = gopt.BezOptimization(**args)
    eng = b._engine(True)
    X = rng.normal(size=(B, b.nvar)) * 3
    L = 2 * deg + E + 1
    P = V * (V - 1) // 2
    nvarN = eng.nvar
    JT = eng.jac_separation(X, E, dense=True).cpu().numpy()
    sw = eng.jac_separation(X, E, dense=False).cpu().numpy()
    assert sw.shape == (B, nvarN * (V - 1), L)
    D = _sweep_to_dense_sep(sw, B, nvarN, V, V, dim, eng.ncols, L, P, -1)
    scale = np.abs(JT).max()
    assert np.abs(D - JT).max() <= 1e-13 * scale
    assert np.array_equal(D == 0, JT == 0)
    JS = eng.jac_speed(X, E, 1.0, dense=True).cpu().numpy()
    ss = eng.jac_speed(X, E, 1.0, dense=False).cpu().numpy()
    assert ss.shape == (B, nvarN, L)
    v_of = np.arange(nvarN) // (dim * eng.ncols)
    for k in range(nvarN):
        assert np.abs(JS[:, k, v_of[k] * L:(v_of[k] + 1) * L] - ss[:, k]).max() <= 1e-13 * np.abs(JS).max()
        mask = np.ones(V * L, dtype=bool)
        mask[v_of[k] * L:(v_of[k] + 1) * L] = False
        assert np.all(JS[:, k, mask] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("nobs,deg,E", [(16, 10, 100), (5, 6, 3), (1, 10, 60)])
def test_one_vehicle_dense_block_is_sweep_block(gopt, batch_mod, nobs, deg, E):
    """one vehicle, npairs = N-1: a point's dense J^T is its sweep block byte for byte"""
    import torch
    probs, sets = _dubins_batch(3, nobs=nobs, deg=deg, seed0=40)
    pb = batch_mod.ProblemBatch(_template(probs[0]), sets)
    eng = pb.eng
    X = _dubins_x(gopt, probs, 4)
    obst = pb.d_obst
    d = eng.jac_separation(X, E, obst_sets=obst, npairs=pb.npairs_x, dense=True)
    s = eng.jac_separation(X, E, obst_sets=obst, npairs=pb.npairs_x, dense=False)
    assert torch.equal(d.reshape(-1), s.reshape(-1))
    d = eng.jac_speed(X, E, -1.0, dense=True)
    s = eng.jac_speed(X, E, -1.0, dense=False)
    assert torch.equal(d.reshape(-1), s.reshape(-1))


@pytest.mark.gpu
@pytest.mark.parametrize("V,obst", [(3, None), (1, [[0.5, -0.5]])])
def test_timeopt_tf_moves_no_control_point(gopt, V, obst):
    """fixed-end time-optimal: tf moves no control point -- its separation row is exactly zero,
    its speed row (the n/tf factor) is not; both match the oracle.  One vehicle and one obstacle:
    the dense block is the sweep block and only the tf row is zero-filled"""
    import torch
    E = 6
    args, rng = _fixed_end(V, 2, 5, 'TimeOpt', 21)
    if obst is not None:
        args["pointObstacles"] = obst
    b = gopt.BezOptimization(**args)
    eng = b._engine(True)
    X = rng.normal(size=(2, b.nvar)) * 3
    X[:, -1] = [9.0, 14.0]
    res = b.jacobian_batch(X, which=BLOCKS, elev=E)
    assert np.all(res["sep"][:, -1].cpu().numpy() == 0)
    assert np.all(np.abs(res["maxspeed"][:, -1].cpu().numpy()).max(axis=1) > 0)
    sw = eng.jac_separation(X, E, dense=False)
    nvarN, N = b.nvar - 1, eng.N
    P = N * (N - 1) // 2
    assert tuple(sw.shape) == (2, nvarN * (N - 1) + P, 2 * 5 + E + 1)
    assert np.all(sw[:, nvarN * (N - 1):].cpu().numpy() == 0)
    if V == 1:
        assert torch.equal(sw.reshape(-1), res["sep"].reshape(-1))
    for i in range(2):
        for name in BLOCKS:
            _check_exact(res[name][i].cpu().numpy().T, _exact(args, X[i], E, name), (i, name))
        single = _single(gopt, args, X[i], E)
        for name in BLOCKS:
            assert np.array_equal(res[name][i].cpu().numpy().T, single[name]), (i, name)


# ---- 4. ProblemBatch.sweep ---------------------------------------------------------------

@pytest.mark.gpu
def test_problem_batch_closed_vs_literal(gopt, batch_mod):
    E = 100
    probs, sets = _dubins_batch(4, nobs=16, deg=10, seed0=60)
    pb = batch_mod.ProblemBatch(_template(probs[0]), sets)
    X = _dubins_x(gopt, probs, 6)
    blocks = ("sep", "maxspeed", "minspeed", "angrate", "sep_closed", "maxspeed_closed", "minspeed_closed",
              "angrate_closed")
    res = pb.sweep(X, elev=E, blocks=blocks)
    assert set(res) == set(blocks)
    for name in BLOCKS:
        f0l, JTl = (t.cpu().numpy() for t in res[name])
        f0c, JTc = (t.cpu().numpy() for t in res[name + "_closed"])
        assert f0c.shape == f0l.shape and JTc.shape == JTl.shape, name
        assert np.array_equal(f0c, f0l), name
        assert np.abs(JTc - JTl).max() / np.abs(JTl).max() < 5e-6, name    # reference FD noise floor
    # the closed blocks alone give the same results as in the mixed call
    alone = pb.sweep(X, elev=E, blocks=("sep_closed",))
    assert np.array_equal(alone["sep_closed"][1].cpu().numpy(), res["sep_closed"][1].cpu().numpy())


# ---- 5. errors ---------------------------------------------------------------------------

@pytest.mark.gpu
def test_errors_on_device(gopt):
    import torch
    from optimalbeziertrajectorygeneration_b200 import _capi, engine
    dev = torch.device("cuda", torch.cuda.current_device())
    buf = torch.zeros(1 << 16, dtype=torch.float64, device=dev)
    p = buf.data_ptr()
    plan = engine.Plan.get(6, 2, 3, dev.index)
    L = 2 * 6 + 3 + 1
    # 1 vehicle + 4 obstacles: P = 10, pairs with the vehicle = 4
    sep = _capi.lib.bez_jac_sepsq_elev_batched
    spd = _capi.lib.bez_jac_speed_sq_elev_batched

    def s(h=plan.handle, cpts=p, B=2, npairs=4, ld=4 * L, dx=p, out=p, kdir=6):
        return sep(h, cpts, B, 5, 1, 3, 2, dx, p, kdir, npairs, 1, out, ld, None)

    def v(h=plan.handle, cpts=p, tf=p, B=2, ld=L, out=p):
        return spd(h, cpts, tf, B, 5, 1, 3, 2, -1.0, p, p, 6, 1, out, ld, None)

    assert s() == 0 and v() == 0
    assert s(B=0) == 0 and v(B=0) == 0
    for bad in (dict(h=None), dict(cpts=None), dict(dx=None), dict(out=None), dict(ld=4 * L - 1),
                dict(npairs=3), dict(npairs=11), dict(B=-1), dict(kdir=2)):
        assert s(**bad) == -1, bad
    for bad in (dict(h=None), dict(cpts=None), dict(tf=None), dict(out=None), dict(ld=L - 1), dict(B=-1)):
        assert v(**bad) == -1, bad
    big = engine.Plan.get(13, 2, 0, dev.index)
    assert s(h=big.handle, ld=4 * 27) == -3
    assert v(h=big.handle, ld=27) == -3
    # the single-point entries: B = 1 over all P = 10 pairs, the same checks
    sep1, spd1 = _capi.lib.bez_jac_sepsq_elev, _capi.lib.bez_jac_speed_sq_elev
    assert sep1(plan.handle, p, 5, 1, 3, 2, p, None, 6, 1, p, 10 * L, None) == 0
    assert spd1(plan.handle, p, 5, 1, 3, 2, 8.0, -1.0, p, None, 6, 1, p, L, None) == 0
    assert sep1(plan.handle, p, 5, 1, 3, 2, p, p, 2, 1, p, 10 * L, None) == -1
    assert spd1(plan.handle, p, 5, 1, 3, 2, 8.0, -1.0, p, p, 2, 1, p, L, None) == -1
    assert sep1(big.handle, p, 5, 1, 3, 2, p, p, 6, 1, p, 10 * 27, None) == -3
    assert spd1(big.handle, p, 5, 1, 3, 2, 8.0, -1.0, p, p, 6, 1, p, 27, None) == -3
    torch.cuda.synchronize()


# ---- CPU: argument validation happens before any CUDA call ---------------------------------

class _FakePlan(ctypes.Structure):
    """Leading fields of bez_plan: the entry points read n, dim and L while validating."""
    _fields_ = [("n", ctypes.c_int), ("dim", ctypes.c_int), ("elev", ctypes.c_int), ("device", ctypes.c_int),
                ("L", ctypes.c_int), ("Lh", ctypes.c_int), ("LhPad", ctypes.c_int), ("ptrs", ctypes.c_void_p * 8)]


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


def test_argument_errors_without_gpu():
    """every rejected argument is rejected on the host: the fake plan's device pointers are never
    touched and no device is needed"""
    _capi = _lib()
    buf = (ctypes.c_double * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    plan = _FakePlan(6, 2, 3, 0, 16, 8, 32)
    big = _FakePlan(13, 2, 0, 0, 27, 14, 32)
    sep = _capi.lib.bez_jac_sepsq_elev_batched
    spd = _capi.lib.bez_jac_speed_sq_elev_batched

    def s(h=ctypes.byref(plan), cpts=p, B=2, npairs=4, ld=4 * 16, dx=p, out=p, N=5):
        return sep(h, cpts, B, N, 1, 3, 2, dx, p, 6, npairs, 1, out, ld, None)

    def v(h=ctypes.byref(plan), cpts=p, tf=p, B=2, ld=16, out=p, dx=p):
        return spd(h, cpts, tf, B, 5, 1, 3, 2, -1.0, dx, p, 6, 1, out, ld, None)

    for bad in (dict(h=None), dict(cpts=None), dict(dx=None), dict(out=None)):
        assert s(**bad) == -1, bad
        assert "NULL" in _capi.last_error()
    for bad in (dict(h=None), dict(cpts=None), dict(tf=None), dict(dx=None), dict(out=None)):
        assert v(**bad) == -1, bad
        assert "NULL" in _capi.last_error()
    assert s(npairs=3) == -1 and "npairs" in _capi.last_error()
    assert s(npairs=11) == -1 and "npairs" in _capi.last_error()
    assert s(ld=4 * 16 - 1) == -1 and "ld" in _capi.last_error()
    assert v(ld=15) == -1 and "ld" in _capi.last_error()
    assert s(B=-1) == -1 and v(B=-1) == -1
    assert s(N=1) == -1
    assert s(h=ctypes.byref(big), ld=4 * 27) == -3
    assert v(h=ctypes.byref(big), ld=27) == -3
    # B = 0 is a no-op (still nothing touches the device)
    assert s(B=0) == 0 and v(B=0) == 0
    # the single-point entries are B = 1 calls with the same checks (all P = 10 pairs)
    sep1, spd1 = _capi.lib.bez_jac_sepsq_elev, _capi.lib.bez_jac_speed_sq_elev

    def s1(h=ctypes.byref(plan), cpts=p, dx=p, out=p, kdir=6, ld=10 * 16):
        return sep1(h, cpts, 5, 1, 3, 2, dx, p, kdir, 1, out, ld, None)

    def v1(h=ctypes.byref(plan), cpts=p, dx=p, out=p, kdir=6, ld=16):
        return spd1(h, cpts, 5, 1, 3, 2, 8.0, -1.0, dx, p, kdir, 1, out, ld, None)

    for f in (s1, v1):
        for bad in (dict(h=None), dict(cpts=None), dict(dx=None), dict(out=None)):
            assert f(**bad) == -1, (f, bad)
            assert "NULL" in _capi.last_error()
        for kdir in (2, 7):
            assert f(kdir=kdir) == -1 and "kdir" in _capi.last_error(), (f, kdir)
    assert s1(ld=10 * 16 - 1) == -1 and "ld" in _capi.last_error()
    assert v1(ld=15) == -1 and "ld" in _capi.last_error()
    assert s1(h=ctypes.byref(big), ld=10 * 27) == -3
    assert v1(h=ctypes.byref(big), ld=27) == -3
