"""Angular-rate Jacobian: literal 2-point sweep vs the closed form (bez_jac_angrate_sq), A/B in one run.

W1  C5 problem batch: M problems (Dubins TimeOpt, n = 10, E = 100, nvar = 15).
    literal = the M x 16 points through bez_angrate_sq + bez_fd_quotient_batched
    closed  = the M base points through bez_angrate_sq + bez_jac_angrate_sq (sweep and dense layout;
              the closed path also computes SciPy's steps on the device, the literal path gets its
              points prebuilt)
    Cold bursts as in tools/ab_pair.py: idle pause, warm-up, then CUDA events around each launch
    sequence; the two paths alternate.  The fp64-pipe share is the DMMA count (SASS of the kernels:
    482 per evaluation, 632 per control-point row, 830 per tf row at U1 = 14) over
    0.25 DMMA/clk/SM x SMs x the maximum SM clock (tools/pipe_bench.cu).
W2  SciPy's closure (B = 1): 2-D Dubins TimeOpt with V vehicles, wall clock per call including the
    synchronising download, literal vs closed alternating.

    python tools/bench_angrate_jac.py --out profiles/r03_angrate_jac.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from optimalbeziertrajectorygeneration_b200 import _capi, engine as _eng, optimization as gopt  # noqa: E402
from optimalbeziertrajectorygeneration_b200.batch import ProblemBatch  # noqa: E402
from oracle.make_golden import dubins_problem_args  # noqa: E402

DMMA_EVAL, DMMA_ROW, DMMA_TF = 482, 632, 830          # U1 = 14 (cuobjdump -sass)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader,nounits", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    name, plim, sm, smmax = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit_w": float(plim), "sm_clock_mhz": float(sm),
            "sm_clock_max_mhz": float(smmax), "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def timed(fn, reps):
    """median / min milliseconds of fn over reps launches, each bracketed by CUDA events"""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out)), float(np.min(out))


def w1(M, rounds, reps, info):
    E = 100
    args = dubins_problem_args(0)
    template = {k: v for k, v in args.items() if k != "pointObstacles"}
    sets = np.repeat(np.asarray(args["pointObstacles"], dtype=np.float64)[None], M, axis=0)
    pb = ProblemBatch(template, sets)
    eng = pb.eng
    rng = np.random.default_rng(0)
    g = np.load(os.path.join(ROOT, "tests", "golden", "constraints.npz"))
    X = g["c5_s0_x"][None] + 0.01 * rng.standard_normal((M, pb.nvar))
    nv1 = pb.nvar + 1
    Xp, dx = pb.fd_points(X)
    Xp = Xp.view(M * nv1, pb.nvar)
    d_X = Xp.view(M, nv1, pb.nvar)[:, 0].contiguous()
    L4 = 4 * (10 + E) + 1
    JT_lit = torch.empty((M, pb.nvar, L4), dtype=torch.float64, device=eng.device)
    ncp = eng.numVeh * 2 * eng.ncols

    def literal():
        F = pb.evaluate(Xp, nv1, E, ("angrate",))["angrate"]
        _capi.call("bez_fd_quotient_batched", _eng._ptr(F), _eng._ptr(dx), M, pb.nvar, L4, _eng._ptr(JT_lit),
                   _eng._stream())

    res = {}

    def closed(dense):
        def run():
            pb.evaluate(d_X, 1, E, ("angrate",))
            res[dense] = eng.jac_angrate_closed(d_X, E, -1.0, dense=dense)
        return run

    paths = {"literal": literal, "closed_sweep": closed(False), "closed_dense": closed(True)}
    for f in paths.values():                     # warm-up: modules, allocations, scratch
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in paths}
    for _ in range(rounds):
        for k, f in paths.items():
            time.sleep(0.5)                      # idle pause: every burst starts cold
            f()
            torch.cuda.synchronize()
            times[k].append(timed(f, reps))
    # accuracy on the timed inputs
    literal()
    jd = res[True]
    jsw = res[False]
    torch.cuda.synchronize()
    rel = float(((jd - JT_lit).abs().amax() / JT_lit.abs().amax()).item())
    dense_vs_sweep = bool(torch.equal(jsw[:, :ncp], jd[:, :ncp, :]) and torch.equal(jsw[:, ncp], jd[:, -1, :]))
    # at the maximum SM clock (the clock read before the run is the idle one): a lower bound of the share
    peak = 0.25 * info["sms"] * info["sm_clock_max_mhz"] * 1e6        # DMMA / s
    dmma = {"literal": M * nv1 * DMMA_EVAL,
            "closed": M * DMMA_EVAL + M * DMMA_EVAL + M * (ncp * DMMA_ROW + DMMA_TF)}
    out = {"M": M, "n": 10, "elev": E, "nvar": pb.nvar, "rounds": rounds, "reps_per_round": reps,
           "max_rel_diff_closed_vs_literal": rel, "sweep_rows_equal_dense": dense_vs_sweep,
           "dmma_model": dmma}
    for k, tl in times.items():
        med = float(np.median([t[0] for t in tl]))
        d = dmma["literal" if k == "literal" else "closed"]
        out[k] = {"median_ms": med, "min_ms": float(np.min([t[1] for t in tl])),
                  "round_medians_ms": [t[0] for t in tl], "fp64_pipe_share_dmma_model": d / peak / (med * 1e-3)}
    out["closed_sweep_over_literal"] = out["closed_sweep"]["median_ms"] / out["literal"]["median_ms"]
    out["closed_dense_over_literal"] = out["closed_dense"]["median_ms"] / out["literal"]["median_ms"]
    return out


def dubins_swarm(V, seed=7):
    rng = np.random.default_rng(seed)
    ia, fa = rng.uniform(-np.pi, np.pi, V), rng.uniform(-np.pi, np.pi, V)
    return dict(numVeh=V, dimension=2, degree=10, minimizeGoal='TimeOpt', maxSep=0.5, maxSpeed=5,
                maxAngRate=1, initPoints=rng.uniform(0, 10 * V ** 0.5, (V, 2)),
                finalPoints=rng.uniform(0, 10 * V ** 0.5, (V, 2)), initSpeeds=np.ones(V), finalSpeeds=np.ones(V),
                initAngs=ia, finalAngs=fa)


def w2(calls, rounds):
    rows = []
    for V in (2, 8, 32):
        for E in (0, 100):
            b = gopt.BezOptimization(**dubins_swarm(V))
            gopt.DEG_ELEV = E
            x = b.generateGuess(std=0.1, seed=1)
            x[-1] = 10.0
            fns = {"literal": b.maxAngularRateConstraints_jac, "closed": b.maxAngularRateConstraints_jac_closed}
            for f in fns.values():
                for _ in range(3):
                    f(x)
            t = {k: [] for k in fns}
            for _ in range(rounds):
                for k, f in fns.items():
                    time.sleep(0.2)
                    ts = []
                    for _ in range(calls):
                        t0 = time.perf_counter()
                        f(x)
                        ts.append(time.perf_counter() - t0)
                    t[k].append(float(np.median(ts)) * 1e3)
            Jl, Jc = fns["literal"](x), fns["closed"](x)
            rows.append({"V": V, "elev": E, "nvar": b.nvar,
                         "literal_ms": float(np.median(t["literal"])), "closed_ms": float(np.median(t["closed"])),
                         "speedup": float(np.median(t["literal"]) / np.median(t["closed"])),
                         "max_rel_diff_closed_vs_literal": float(np.abs(Jc - Jl).max() / np.abs(Jl).max())})
            print(json.dumps(rows[-1]), flush=True)
    gopt.DEG_ELEV = 0
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_angrate_jac.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    r1 = w1(a.M, a.rounds, a.reps, info)
    print(json.dumps(r1), flush=True)
    r2 = w2(a.calls, a.rounds)
    info_after = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"device": info, "device_after": info_after, "W1_c5_batch": r1, "W2_closure": r2}, f, indent=1)


if __name__ == "__main__":
    main()
