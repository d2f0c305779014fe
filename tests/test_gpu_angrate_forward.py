"""Forward values of the angular-rate block (bez_angrate_sq, ConstraintEngine.angrate,
BezOptimization.maxAngularRateConstraints) for every kernel generation:

  angrate_mma_kernel<U1>   default for m = n + E <= 127, one instantiation per U1 = ceil((m+1)/8)
  angrate_warp2_kernel     BEZGPU_ANGRATE_GEN=3 (m <= 127)
  angrate_warp_kernel      BEZGPU_ANGRATE_GEN=2 (m <= 127)
  angrate_kernel           the only kernel for 127 < m <= 250; BEZGPU_ANGRATE_V1=1 forces it for every m

Judged against the oracle's restatement of the reference evaluated in 80-bit long double on the
fp64 inputs and tables (about 1e-16 from the exact rational result; test_long_double_oracle_is_exact
checks that).  Bar: block-relative 1e-9, the project's contract for every constraint block, and the
same bound per vehicle row so that a slow-turning vehicle is not hidden behind a fast one.

Every generation lands about 1e-11 from the oracle at m = 127 (measured on an NVIDIA B200 at a 1000 W power limit: worst
block-relative 1.2e-11, per row 2.2e-11), as does the reference's own fp64 evaluation: the worst
entries are the end coefficients, whose x'' is a second difference of elevated control points
that lie about 1/m apart, so fp64 rounding of those points is amplified by about m^2."""
import ctypes

import numpy as np
import pytest

TOL = 1e-9                   # block-relative and per vehicle row
GUARD_IF_TIGHT = 1e-11       # per-row regression guard once a sweep's worst block error is <= 1e-13
LD = np.longdouble
needs_long_double = pytest.mark.skipif(
    np.finfo(np.longdouble).nmant < 63,
    reason="np.longdouble is not the 80-bit extended format here; the oracle would be no better than fp64")

# every bit pattern the kernels could leave behind is distinguishable from this NaN payload
FILL = np.uint64(0x7FF4DEAD0000BEEF)
HALO = 64                    # guard doubles before and after every output buffer

GENS = {"default": {}, "gen3": {"BEZGPU_ANGRATE_GEN": "3"}, "gen2": {"BEZGPU_ANGRATE_GEN": "2"},
        "v1": {"BEZGPU_ANGRATE_V1": "1"}}


@pytest.fixture(scope="module")
def gopt():
    import torch
    assert torch.cuda.is_available()
    from optimalbeziertrajectorygeneration_b200 import optimization
    yield optimization
    optimization.DEG_ELEV = 0


def _use_gen(monkeypatch, gen):
    monkeypatch.delenv("BEZGPU_ANGRATE_GEN", raising=False)
    monkeypatch.delenv("BEZGPU_ANGRATE_V1", raising=False)
    for k, v in GENS[gen].items():
        monkeypatch.setenv(k, v)


# ---- inputs ----------------------------------------------------------------------------------

def _arc(n, rng):
    """[2, n+1] control points on a circular arc that turns by less than a right angle, unevenly
    spaced: every leg of the control polygon, and so every (elevated) first-derivative control
    point, lies within 90 degrees of every other, so all Bernstein coefficients of x'^2 + y'^2 are
    positive and the control-point-wise ratio is well conditioned; the curvature is not zero."""
    R = rng.uniform(2.0, 6.0)
    th = rng.uniform(0, 2 * np.pi) + rng.choice([-1, 1]) * rng.uniform(0.6, 1.3) * \
        (np.arange(n + 1) / n) ** rng.uniform(0.8, 1.25)
    c = rng.uniform(-3, 3, size=2)
    return np.stack([c[0] + R * np.cos(th), c[1] + R * np.sin(th)])


_NS = (2, 3, 5, 10, 16)


def _shape(m, nveh=2):
    """Deterministic (n, E, rows [nveh, 2(n+1)], tf) of degree m = n + E; n cycles through _NS.
    m = 1 is a straight segment (n = 1, E = 0) with small-integer coordinates and val = m/tf = 2,
    so that every product is exact and x'' is exactly 0 in every kernel: the ratio must be 0."""
    if m == 1:
        rows = np.array([[0.0, 3.0, 0.0, 1.0], [1.0, -2.0, 5.0, 4.0]])[:nveh]
        return 1, 0, rows, 0.5
    n = _NS[m % len(_NS)]
    if n > m:
        n = 5
    rng = np.random.default_rng(1000 + m)
    rows = np.stack([_arc(n, rng).reshape(-1) for _ in range(nveh)])
    return n, m - n, rows, float(rng.uniform(1.5, 9.0))


def _pack(rows, B=1, N=None, pad=2):
    """vehicle rows [B or 1, nveh, 2(n+1)] -> cpts [B, N, 2(n+1) + pad]: padding and the rows past
    the vehicles (obstacles) hold NaN, so a kernel that reads them poisons its output."""
    rows = np.asarray(rows, dtype=np.float64)
    if rows.ndim == 2:
        rows = np.broadcast_to(rows, (B,) + rows.shape)
    B, nveh, w = rows.shape
    N = nveh if N is None else N
    cpts = np.full((B, N, w + pad), np.nan)
    cpts[:, :nveh, :w] = rows
    return cpts


def _run(n, E, cpts, tf, alpha=1.0, beta=0.0, veh_begin=0, nveh=None, b0=0, B=None):
    """bez_angrate_sq on host cpts [Btot, N, S] and tf [Btot] for points b0 .. b0+B-1 and vehicles
    veh_begin .. veh_begin+nveh-1 -> host [B, nveh, 4m+1].  The output buffer starts out as a NaN
    payload no kernel produces, with HALO guard doubles on both sides: every entry must be
    written, and nothing before or after it."""
    import torch
    from optimalbeziertrajectorygeneration_b200 import _capi, engine
    cpts = np.ascontiguousarray(cpts, dtype=np.float64)
    tf = np.array(np.broadcast_to(np.asarray(tf, dtype=np.float64), cpts.shape[:1]))
    Btot, N, S = cpts.shape
    B = Btot - b0 if B is None else B
    nveh = N - veh_begin if nveh is None else nveh
    size = B * nveh * (4 * (n + E) + 1)
    tabs = engine.AngRateTables.get(n, E, torch.cuda.current_device())
    d_c = torch.from_numpy(cpts).cuda()
    d_tf = torch.from_numpy(tf).cuda()
    d_out = torch.from_numpy(np.full(size + 2 * HALO, FILL, dtype=np.uint64).view(np.float64)).cuda()
    _capi.call("bez_angrate_sq", tabs.handle, ctypes.c_void_p(d_c.data_ptr() + 8 * b0 * N * S),
               ctypes.c_void_p(d_tf.data_ptr() + 8 * b0), B, N, S, veh_begin, nveh, float(alpha),
               float(beta), ctypes.c_void_p(d_out.data_ptr() + 8 * HALO),
               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    got = d_out.cpu().numpy()
    bits = got.view(np.uint64)
    assert np.all(bits[:HALO] == FILL) and np.all(bits[HALO + size:] == FILL), "wrote outside the output"
    unwritten = int(np.count_nonzero(bits[HALO:HALO + size] == FILL))
    assert unwritten == 0, "%d of %d output entries not written" % (unwritten, size)
    return got[HALO:HALO + size].reshape(B, nveh, -1)


# ---- oracle -----------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def oracle():
    """ratio(n, E, rows [B, nveh, 2(n+1)], tf [B]) -> long-double squared angular rate
    [B, nveh, 4m+1]; rows are cached per (shape, input), so every generation reuses them."""
    from oracle import bezier_oracle as O
    cache = {}

    def ratio(n, E, rows, tf):
        rows = np.asarray(rows, dtype=np.float64)
        if rows.ndim == 2:
            rows = rows[None]
        tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), rows.shape[:1])
        out = []
        for b in range(rows.shape[0]):
            for v in range(rows.shape[1]):
                key = (n, E, rows[b, v].tobytes(), float(tf[b]))
                if key not in cache:
                    pos = O.elev(rows[b, v].reshape(2, n + 1), E, dtype=LD)
                    cache[key] = O.angular_rate_sq(pos, float(tf[b]), dtype=LD)
                out.append(cache[key])
        return np.array(out, dtype=LD).reshape(rows.shape[:2] + (-1,))

    return ratio


def _errors(got, want):
    """(worst block-relative error over the points, worst per-row relative error) of got [B, nveh, L]
    against want (long double); a block is one evaluation point's rows."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.all(np.isfinite(got)), "non-finite output where the reference is finite"
    d = np.abs(got.astype(LD) - want)
    a = np.abs(want)
    blk = d.max(axis=(1, 2)) / np.maximum(a.max(axis=(1, 2)), 1e-300)
    row = d.max(axis=2) / np.maximum(a.max(axis=2), 1e-300)
    return float(blk.max()), float(row.max())


class _Sweep:
    """Worst errors over a sweep, and one line per shape for the report."""

    def __init__(self, name):
        self.name, self.blk, self.row, self.bad = name, 0.0, 0.0, []

    def add(self, label, got, want):
        blk, row = _errors(got, want)
        self.blk, self.row = max(self.blk, blk), max(self.row, row)
        if blk > TOL or row > TOL:
            self.bad.append("%s: block %.2e, row %.2e" % (label, blk, row))

    def finish(self):
        print("\n%s: worst block-relative %.2e, worst per-row %.2e" % (self.name, self.blk, self.row))
        assert not self.bad, "above the %g bar:\n  %s" % (TOL, "\n  ".join(self.bad))
        if self.blk <= 1e-13:
            assert self.row <= GUARD_IF_TIGHT, (self.name, self.row)


# ---- a. every instantiation of the default kernel ---------------------------------------------

SWEEP_M = [m for u in range(1, 17) for m in (8 * u - 8, 8 * u - 1) if m > 0]     # both ends of every U1


def test_sweep_covers_every_instantiation():
    assert len(SWEEP_M) == 31
    assert sorted({(m + 8) // 8 for m in SWEEP_M}) == list(range(1, 17))


@needs_long_double
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_default_every_instantiation(gopt, oracle, monkeypatch):
    """angrate_mma_kernel<U1> for U1 = 1..16 at both ends of each bucket.  Even positions go through
    the C-ABI (raw ratio: alpha = 1, beta = 0), odd ones through BezOptimization (alpha = -1,
    beta = maxAngRate^2), compared with maxAngRate^2 - ratio of the oracle."""
    _use_gen(monkeypatch, "default")
    sw = _Sweep("angrate_mma_kernel (default, m <= 127)")
    for i, m in enumerate(SWEEP_M):
        n, E, rows, tf = _shape(m)
        want = oracle(n, E, rows, tf)
        if i % 2 == 0:
            got = _run(n, E, _pack(rows), tf)
        else:
            maxrate = 0.5
            b = gopt.BezOptimization(numVeh=rows.shape[0], dimension=2, degree=n, minimizeGoal='Euclidean',
                                     maxAngRate=maxrate, tf=tf)
            gopt.DEG_ELEV = E
            got = b.maxAngularRateConstraints(rows.reshape(-1)).reshape(want.shape)
            want = LD(maxrate) ** 2 - want
        sw.add("m %d (n %d, E %d)" % (m, n, E), got, want)
    sw.finish()


# ---- b. first generation above the tensor path -------------------------------------------------

@needs_long_double
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_first_generation_above_127(oracle, monkeypatch):
    _use_gen(monkeypatch, "default")
    sw = _Sweep("angrate_kernel (m > 127)")
    for m in (128, 129, 136, 160, 200, 239, 240, 249, 250):
        n, E, rows, tf = _shape(m)
        sw.add("m %d (n %d, E %d)" % (m, n, E), _run(n, E, _pack(rows), tf), oracle(n, E, rows, tf))
    sw.finish()


# ---- c. forced generations ---------------------------------------------------------------------

@needs_long_double
@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("gen", ["gen3", "gen2", "v1"])
def test_forced_generation(oracle, monkeypatch, gen):
    _use_gen(monkeypatch, gen)
    sw = _Sweep("%s (m <= 127)" % gen)
    for m in (1, 7, 8, 63, 64, 110, 127):
        n, E, rows, tf = _shape(m)
        sw.add("m %d (n %d, E %d)" % (m, n, E), _run(n, E, _pack(rows), tf), oracle(n, E, rows, tf))
    sw.finish()


# ---- d. layout through the C-ABI ---------------------------------------------------------------

# numVeh = 13 vehicles + 2 obstacle rows, B = 3 points with their own tf (a time-optimal model)
LAYOUT_TF = (2.0, 3.75, 7.125)


def _layout_inputs(n, numVeh=13, B=3, seed=7):
    rng = np.random.default_rng(seed)
    rows = np.stack([np.stack([_arc(n, rng).reshape(-1) for _ in range(numVeh)]) for _ in range(B)])
    return rows, _pack(rows, N=numVeh + 2)


@needs_long_double
@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("gen,n,E", [("default", 5, 19), ("gen3", 5, 19), ("gen2", 5, 19), ("v1", 5, 19),
                                     ("default", 3, 129)])
def test_layout(oracle, monkeypatch, gen, n, E):
    """Points, vehicle sub-ranges, partial blocks, padded rows: sub-launches write exactly the rows
    of the full launch, bit for bit; B * nveh = 1, 3, 5, 13 and 15 leave the last block of four
    warps partial (39 for the full launch)."""
    _use_gen(monkeypatch, gen)
    rows, cpts = _layout_inputs(n)
    B, numVeh = rows.shape[:2]
    full = _run(n, E, cpts, LAYOUT_TF, veh_begin=0, nveh=numVeh)
    if E < 100:                                   # the oracle for 39 vehicles at m = 132 would take minutes
        sw = _Sweep("layout %s m %d" % (gen, n + E))
        sw.add("full launch", full, oracle(n, E, rows, LAYOUT_TF))
        sw.finish()
    else:
        sw = _Sweep("layout %s m %d (sample)" % (gen, n + E))
        sw.add("point 1, vehicles 11..12", full[1:2, 11:], oracle(n, E, rows[1:2, 11:], LAYOUT_TF[1]))
        sw.finish()
    for b0, nb, vb, nv in ((2, 1, 6, 1), (0, 3, 12, 1), (2, 1, 3, 5), (1, 1, 0, 13), (0, 3, 1, 5), (1, 2, 4, 4)):
        sub = _run(n, E, cpts, LAYOUT_TF, veh_begin=vb, nveh=nv, b0=b0, B=nb)
        ref = full[b0:b0 + nb, vb:vb + nv]
        assert sub.tobytes() == ref.tobytes(), (b0, nb, vb, nv)
    # a NaN control point makes exactly its vehicle's rows NaN; every other row keeps its bits
    cpts[1, 4, 3] = np.nan
    poisoned = _run(n, E, cpts, LAYOUT_TF, veh_begin=0, nveh=numVeh)
    assert np.all(np.isnan(poisoned[1, 4]))
    keep = np.ones((B, numVeh), dtype=bool)
    keep[1, 4] = False
    assert poisoned[keep].tobytes() == full[keep].tobytes()


# ---- e. unit changes ---------------------------------------------------------------------------

UNIT_CASES = [(g, m) for g in ("default", "gen3", "gen2", "v1") for m in (8, 64, 110, 127)] + \
             [("default", m) for m in (128, 200, 240, 250)]


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("gen,m", UNIT_CASES)
def test_unit_changes(monkeypatch, gen, m):
    """The squared angular rate does not depend on the spatial unit and scales as tf^-2.  Every
    operation of the kernels is scale-equivariant, so in fp64 (away from overflow and underflow)
    control points x 2^k must leave the raw ratio bit-identical, and tf x 2^j must multiply it by
    exactly 2^(-2j).  That includes the tensor-path kernel's rcp.approx division and its Newton
    steps.  At m = 250, cpts x 2^16 is a change from metres to about centimetres; before the
    first-generation kernel rescaled its degree-2m rows, it and tf x 2^-8 overflowed there."""
    _use_gen(monkeypatch, gen)
    n, E, rows, tf = _shape(m)
    base = _run(n, E, _pack(rows), tf)
    assert np.all(np.isfinite(base))
    bad = []
    for k in (-40, -16, -4, 4, 16, 40):
        got = _run(n, E, _pack(np.ldexp(rows, k)), tf)
        if got.tobytes() != base.tobytes():
            bad.append("cpts x 2^%d: %d non-finite, %d differ" % (
                k, np.count_nonzero(~np.isfinite(got)), np.count_nonzero(got != base)))
    for j in (-8, -2, 2, 8):
        got = _run(n, E, _pack(rows), np.ldexp(tf, j))
        want = np.ldexp(base, -2 * j)
        if got.tobytes() != want.tobytes():
            bad.append("tf x 2^%d: %d non-finite, %d differ" % (
                j, np.count_nonzero(~np.isfinite(got)), np.count_nonzero(got != want)))
    assert not bad, "%s m %d: %s" % (gen, m, "; ".join(bad))


# ---- f. degenerate inputs ----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("gen", list(GENS))
def test_degree_one_is_exactly_beta(monkeypatch, gen):
    """n = 1, E = 0: x'' is 0, so alpha * ratio + beta is exactly beta.  In the reference x'' is
    exactly 0; the kernels' derivative stencil p_{k+1} val - p_k val may be contracted into one
    FMA, which leaves at most the rounding error of one product, so the raw ratio is 0 or of the
    order of (eps val)^2 (val = m/tf)."""
    _use_gen(monkeypatch, gen)
    rng = np.random.default_rng(11)
    rows = rng.uniform(-5, 5, size=(3, 4))
    tf = (1.7, 3.3)
    got = _run(1, 0, _pack(rows, B=2), tf, alpha=-1.0, beta=0.7)
    assert got.shape == (2, 3, 5)
    assert np.all(got == 0.7)
    raw = _run(1, 0, _pack(rows, B=2), tf)
    assert np.all(np.abs(raw) <= 1e-28 / np.square(tf)[:, None, None])
    print("\n%s: %d of %d raw ratios exactly 0, largest %.1e" % (gen, np.count_nonzero(raw == 0), raw.size,
                                                                np.abs(raw).max()))


@needs_long_double
@pytest.mark.gpu
@pytest.mark.parametrize("gen,E", [("default", 20), ("gen3", 20), ("gen2", 20), ("v1", 20), ("default", 140)])
def test_straight_next_to_curved(oracle, monkeypatch, gen, E):
    """A straight vehicle (a segment elevated to degree n) in the same launch as a curved one: its
    rate is rounding noise in the oracle and in the kernel alike, far below the block's scale."""
    from oracle import bezier_oracle as O
    _use_gen(monkeypatch, gen)
    n = 5
    rng = np.random.default_rng(12)
    straight = O.elev(np.array([[-1.25, 4.5], [0.5, -2.0]]), n - 1)
    rows = np.stack([_arc(n, rng).reshape(-1), straight.reshape(-1)])
    got = _run(n, E, _pack(rows), 2.5)
    want = oracle(n, E, rows, 2.5)
    blk = float(np.abs(got.astype(LD) - want).max() / np.abs(want).max())
    assert blk <= TOL
    assert _errors(got[:, :1], want[:, :1])[1] <= TOL
    assert np.abs(got[0, 1]).max() <= TOL * np.abs(want).max()


@needs_long_double
@pytest.mark.gpu
@pytest.mark.parametrize("gen", list(GENS))
def test_stationary_vehicle_is_nan(monkeypatch, gen):
    """All control points equal: x' = x'' = 0, every coefficient is 0/0 as in the reference.  The
    points sit at the origin (any E) or, at E = 0, elsewhere with m/tf = 2 so that the
    derivative stencil is exact whichever way it is rounded."""
    from oracle import bezier_oracle as O
    _use_gen(monkeypatch, gen)
    n = 6
    rows = np.stack([np.zeros(2 * (n + 1)), np.repeat([1.25, -3.5], n + 1), _arc(n, np.random.default_rng(13)).ravel()])
    for E, tf in ((0, n / 2.0), (30, 2.5)):
        got = _run(n, E, _pack(rows if E == 0 else rows[[0, 2]]), tf)
        assert np.all(np.isnan(got[0, 0]))
        with np.errstate(invalid="ignore", divide="ignore"):
            assert np.all(np.isnan(O.angular_rate_sq(O.elev(rows[0].reshape(2, -1), E), tf)))
        if E == 0:
            assert np.all(np.isnan(got[0, 1]))
        assert np.all(np.isfinite(got[0, -1]))


@needs_long_double
@pytest.mark.gpu
@pytest.mark.parametrize("gen,n", [("default", 5), ("default", 10), ("default", 16), ("gen3", 10),
                                   ("gen2", 10), ("v1", 10), ("default", 136)])
def test_start_from_rest(oracle, monkeypatch, gen, n):
    """Control point 1 equals control point 0 (E = 0, m/tf = 2 so that x'_0 is exactly 0 in the
    kernels and in the reference): the first four coefficients of DEN^2 vanish.  So do those of
    NUM^2 in the reference, whose num_1 = y''_0 x'_1 - x''_0 y'_1 = 2 (y'_1 x'_1 - x'_1 y'_1) is
    exactly 0, so numpy gives NaN (0/0) at all four.  Kernels that fuse those products into FMAs
    leave a rounding residue in num_1 and give +inf (residue/0) at two of them (on a B200: the
    warp kernels at n = 10 and the first generation at n = 136); the tensor-path kernel's
    reciprocal makes every x/0 a NaN.  Wherever the fp64 reference is non-finite the kernel must
    be too; every other entry meets the bar."""
    from oracle import bezier_oracle as O
    _use_gen(monkeypatch, gen)
    rng = np.random.default_rng(14)
    rows = np.stack([_arc(n, rng) for _ in range(2)])
    rows[0, :, 1] = rows[0, :, 0]
    rows = rows.reshape(2, -1)
    tf = n / 2.0
    got = _run(n, 0, _pack(rows), tf)[0]
    with np.errstate(invalid="ignore", divide="ignore"):
        ref64 = np.stack([O.angular_rate_sq(r.reshape(2, -1), tf) for r in rows])
        want = oracle(n, 0, rows, tf)[0]
    bad = ~np.isfinite(ref64)
    assert list(np.flatnonzero(bad[0])) == [0, 1, 2, 3] and not bad[1].any()
    assert np.all(np.isnan(ref64[bad]))
    assert np.all(~np.isfinite(got[bad]))
    print("\n%s n %d: fp64 reference nan %d inf %d; kernel nan %d inf %d" % (
        gen, n, np.isnan(ref64).sum(), np.isinf(ref64).sum(), np.isnan(got[bad]).sum(), np.isinf(got[bad]).sum()))
    ok = ~bad
    assert np.all(np.isfinite(want[ok]))
    d = np.abs(got[ok].astype(LD) - want[ok])
    assert float(d.max() / np.abs(want[ok]).max()) <= TOL
    assert _errors(got[1:2][None], want[1:2][None])[1] <= TOL


# ---- g. limits and the literal Jacobian above the tensor path -----------------------------------

@pytest.mark.gpu
def test_degree_251_is_refused(gopt):
    from optimalbeziertrajectorygeneration_b200 import _capi
    b = gopt.BezOptimization(numVeh=1, dimension=2, degree=5, minimizeGoal='Euclidean', tf=2.0)
    gopt.DEG_ELEV = 246
    with pytest.raises(_capi.BezGpuError, match="250"):
        b.maxAngularRateConstraints(_arc(5, np.random.default_rng(15)).ravel())


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_literal_jacobian_m200_matches_forward_calls(gopt):
    """Above the tensor path the angular-rate Jacobian is the literal quotient of one batched
    launch; it must equal SciPy's quotient formed from separate forward calls, bit for bit."""
    from oracle import bezier_oracle as O
    rng = np.random.default_rng(16)
    args = dict(numVeh=2, dimension=2, degree=8, minimizeGoal='TimeOpt', maxAngRate=2.0,
                initPoints=rng.uniform(-5, 5, size=(2, 2)), finalPoints=rng.uniform(-5, 5, size=(2, 2)))
    b = gopt.BezOptimization(**args)
    x = b.generateGuess(std=0.3, seed=3)
    x[-1] = 4.0
    gopt.DEG_ELEV = 192
    J = b.maxAngularRateConstraints_jac(x)
    f0 = b.maxAngularRateConstraints(x)
    assert np.all(np.isfinite(f0))
    h, dx = O.fd_steps(x)
    for k in (0, x.size // 2, x.size - 1):
        x1 = x.copy()
        x1[k] = x[k] + h[k]
        q = (b.maxAngularRateConstraints(x1) - f0) / dx[k]
        assert q.tobytes() == J[:, k].tobytes(), k


# ---- CPU ------------------------------------------------------------------------------------------

@needs_long_double
@pytest.mark.parametrize("n,E", [(5, 3), (10, 30)])
def test_long_double_oracle_is_exact(n, E):
    """The yardstick: the long-double oracle agrees with the rational one (exact on the fp64 inputs
    and tables) to 1e-15 of the block at m = 8 and 40."""
    from fractions import Fraction
    from oracle import bezier_oracle as O
    c = _arc(n, np.random.default_rng(17))
    tf = 3.7
    exact = O.angular_rate_sq(O.elev(c, E, dtype=object), tf, dtype=object)
    ld = O.angular_rate_sq(O.elev(c, E, dtype=LD), tf, dtype=LD)
    err = max(abs(Fraction(*v.as_integer_ratio()) - r) for v, r in zip(ld, exact))
    assert float(err / max(abs(r) for r in exact)) <= 1e-15


def test_degree_251_is_refused_without_gpu():
    """The degree limit is checked before any CUDA call, and no tables come back."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "optimalbeziertrajectorygeneration_b200", "libbezgpu.so")):
        sys.path.insert(0, root)
        import __graft_entry__ as g
        g.build()
    from optimalbeziertrajectorygeneration_b200 import _capi
    buf = (ctypes.c_double * 4)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    out = ctypes.c_void_p(0)
    assert _capi.lib.bez_angrate_tables_create(10, 241, 0, p, p, p, p, ctypes.byref(out)) == -3
    assert "250" in _capi.last_error()
    assert not out.value
