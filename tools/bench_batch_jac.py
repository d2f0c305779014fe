"""Batched closed-form separation / speed Jacobians vs the literal 2-point sweep, A/B in one run.

W1  C5 problem batch (bench.py's C5 template and seeds: Dubins TimeOpt, 1 vehicle, 16 obstacles,
    n = 10, E = 100, nvar = 15).  Per block, device work only (points and divisors prebuilt):
      literal = the M x 16 points through the constraint kernel + bez_fd_quotient_batched
      closed  = the M base points assembled once, f0 there + bez_jac_*_batched
    and whole ProblemBatch.sweep calls (host X in, fd_points included) for three block sets.
    Cold bursts as in tools/bench_angrate_jac.py: idle pause, warm-up, then CUDA events around each
    launch sequence; the paths alternate.  The separation block's HBM fraction is its algorithmic
    bytes (computed below from the shapes) over the median time, against 6484.6 GB/s (the
    project's measured copy bandwidth, DESIGN section 5).
W2  Single-point C4 separation sweep (tools/prof_jac.py's shape, the 27 GB block) and the C4 speed
    sweep, timed for this build and -- with --parent-root, a checkout of the parent commit with its
    library built -- for that build, in alternating worker processes.  The workers also report
    checksums of the C4 outputs and write Example1's dense Jacobians (E = 0, 10), so the two
    builds' single-point results are compared bit for bit.

    python tools/bench_batch_jac.py --out profiles/r04_batch_jac.json [--parent-root DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM_GBS = 6484.6


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader,nounits", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    name, plim, sm, smmax = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit_w": float(plim), "sm_clock_mhz": float(sm),
            "sm_clock_max_mhz": float(smmax), "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def timed(fn, reps):
    """median / min milliseconds of fn over reps launch sequences, each bracketed by CUDA events"""
    import torch
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out)), float(np.min(out))


def ab(paths, rounds, reps):
    import torch
    for f in paths.values():                     # warm-up: modules, allocations
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in paths}
    for _ in range(rounds):
        for k, f in paths.items():
            time.sleep(0.5)                      # idle pause: every burst starts cold
            f()
            torch.cuda.synchronize()
            times[k].append(timed(f, reps))
    return {k: {"median_ms": float(np.median([t[0] for t in tl])), "min_ms": float(np.min([t[1] for t in tl])),
                "round_medians_ms": [t[0] for t in tl]} for k, tl in times.items()}


def c5_inputs(M):
    """bench.py c5_measure's template, obstacle sets and points (seeds per problem)"""
    from optimalbeziertrajectorygeneration_b200 import optimization as gopt
    deg, nobs = 10, 16
    template = dict(numVeh=1, dimension=2, degree=deg, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=3,
                    maxAngRate=np.pi / 2, initPoints=[(0, 0)], finalPoints=[(12, 8)], initSpeeds=[1],
                    finalSpeeds=[1], tf=8, initAngs=[np.pi / 2], finalAngs=[0])
    sets = np.stack([np.random.default_rng(p).uniform(1.0, 11.0, size=(nobs, 2)) for p in range(M)])
    guess = gopt.BezOptimization(**template).generateGuess(std=0)
    X = guess[None, :] + np.stack([np.random.default_rng(10 ** 6 + p).normal(size=guess.size) * 0.5
                                   for p in range(M)])
    X[:, -1] = np.abs(X[:, -1]) + 4.0
    return template, sets, X


def sep_bytes(M, N, S, nvar, npairs, L):
    """algorithmic HBM bytes of the separation block (f0 + J^T) of one sweep"""
    nv1 = nvar + 1
    literal = 8 * (M * nv1 * N * S                 # control-point rows read
                   + M * nv1 * npairs * L          # rows written
                   + M * nv1 * npairs * L          # rows read back by the quotient kernel
                   + M * nvar * npairs * L)        # J^T written
    closed = 8 * (M * nvar * npairs * L + M * npairs * L + M * N * S)
    return literal, closed


def w1(M, rounds, reps):
    import torch
    from optimalbeziertrajectorygeneration_b200 import _capi, engine as _eng
    from optimalbeziertrajectorygeneration_b200.batch import ProblemBatch
    E = 100
    template, sets, X = c5_inputs(M)
    pb = ProblemBatch(template, sets)
    eng, m = pb.eng, pb.model
    nv1, nvar = pb.nvar + 1, pb.nvar
    L = 2 * 10 + E + 1
    Xp, dx = pb.fd_points(X)
    Xp = Xp.view(M * nv1, nvar)
    d_X = Xp.view(M, nv1, nvar)[:, 0].contiguous()
    JT = {k: torch.empty((M, nvar, w), dtype=torch.float64, device=eng.device)
          for k, w in (("sep", pb.npairs_x * L), ("maxspeed", L))}
    JC = {k: torch.empty_like(v) for k, v in JT.items()}

    def literal(block):
        def run():
            F = pb.evaluate(Xp, nv1, E, (block,))[block]
            _capi.call("bez_fd_quotient_batched", _eng._ptr(F), _eng._ptr(dx), M, nvar, int(F.shape[1]),
                       _eng._ptr(JT[block]), _eng._stream())
        return run

    def closed(block):
        def run():
            cpts, tf = eng.assemble(d_X, E, obst_sets=pb.d_obst, evals_per_set=1)
            base = (cpts, tf, dx, True)
            if block == "sep":
                eng.separation(cpts, E, m["maxSep"], pair_begin=0, npairs=pb.npairs_x)
                eng.jac_separation(None, E, npairs=pb.npairs_x, out=JC[block], base=base)
            else:
                eng.speed(cpts, tf, E, -1.0, float(m["maxSpeed"]) ** 2)
                eng.jac_speed(None, E, -1.0, out=JC[block], base=base)
        return run

    cpts0, tf0 = eng.assemble(d_X, E, obst_sets=pb.d_obst, evals_per_set=1)

    def closed_jac_only():
        eng.jac_separation(None, E, npairs=pb.npairs_x, out=JC["sep"], base=(cpts0, tf0, dx, True))

    blocks = ab({"sep_literal": literal("sep"), "sep_closed": closed("sep"), "sep_closed_jacobian_kernel_only":
                 closed_jac_only, "maxspeed_literal": literal("maxspeed"), "maxspeed_closed": closed("maxspeed")},
                rounds, reps)
    torch.cuda.synchronize()
    rel = {k: float(((JC[k] - JT[k]).abs().amax() / JT[k].abs().amax()).item()) for k in JT}
    sweeps = {"literal_sep_maxspeed_angrate": ("sep", "maxspeed", "angrate"),
              "closed_sep_maxspeed_literal_angrate": ("sep_closed", "maxspeed_closed", "angrate"),
              "all_closed": ("sep_closed", "maxspeed_closed", "angrate_closed")}
    sw = ab({k: (lambda b=b: pb.sweep(X, elev=E, blocks=b)) for k, b in sweeps.items()}, rounds, max(2, reps // 2))
    lit_b, cl_b = sep_bytes(M, eng.N, eng.row_stride, nvar, pb.npairs_x, L)
    out = {"M": M, "n": 10, "elev": E, "nvar": nvar, "N": eng.N, "npairs_x": pb.npairs_x, "L": L,
           "rounds": rounds, "reps_per_round": reps, "blocks": blocks, "sweeps": sw,
           "sweep_block_sets": {k: list(v) for k, v in sweeps.items()},
           "max_rel_diff_closed_vs_literal": rel,
           "sep_algorithmic_bytes": {"literal": lit_b, "closed": cl_b},
           "sep_hbm_fraction_of_%.1f_GBs" % HBM_GBS: {
               "literal": lit_b / (blocks["sep_literal"]["median_ms"] * 1e-3) / 1e9 / HBM_GBS,
               "closed": cl_b / (blocks["sep_closed"]["median_ms"] * 1e-3) / 1e9 / HBM_GBS}}
    out["sep_closed_speedup"] = blocks["sep_literal"]["median_ms"] / blocks["sep_closed"]["median_ms"]
    out["maxspeed_closed_speedup"] = blocks["maxspeed_literal"]["median_ms"] / blocks["maxspeed_closed"]["median_ms"]
    return out


# ---- W2: one build per worker process ---------------------------------------------------------------

def checksum(t):
    """order-dependent checksum of a float64 tensor's bits (wrapping int64 arithmetic, chunked)"""
    import torch
    v = t.reshape(-1).view(torch.int64)
    s1 = s2 = 0
    step = 1 << 26
    for i in range(0, v.numel(), step):
        c = v[i:i + step]
        w = torch.arange(i, i + c.numel(), device=c.device, dtype=torch.int64) % 1000003 + 1
        s1 = (s1 + int(c.sum().item())) & ((1 << 64) - 1)
        s2 = (s2 + int((c * w).sum().item())) & ((1 << 64) - 1)
    return "%016x%016x" % (s1, s2)


def worker(reps, dump_dir):
    import torch
    from bench import WORKLOAD, synthetic_swarm
    from optimalbeziertrajectorygeneration_b200 import optimization as gopt
    res = {}
    if dump_dir:                                    # Example1 dense, E = 0 and 10
        ex1 = dict(numVeh=2, dimension=2, degree=10, minimizeGoal='TimeOpt', maxSep=1, maxSpeed=5, maxAngRate=1,
                   initPoints=[(0, 5), (3, 0)], finalPoints=[(8, 4), (7, 10)], initSpeeds=[1, 1],
                   finalSpeeds=[1, 1], initAngs=[0, np.pi / 2], finalAngs=[0, np.pi / 2], tf=10,
                   pointObstacles=[[3, 2], [6, 7]])
        b = gopt.BezOptimization(**ex1)
        x = b.generateGuess(std=0.3, seed=5)
        for E in (0, 10):
            e1, e0 = b._engine(True), b._engine(False)
            np.save(os.path.join(dump_dir, "ex1_sep_E%d.npy" % E), e1.jac_separation(x, E, dense=True).cpu().numpy())
            np.save(os.path.join(dump_dir, "ex1_speed_E%d.npy" % E), e0.jac_speed(x, E, -1.0).cpu().numpy())
    N, deg, E = WORKLOAD["N"], WORKLOAD["deg"], WORKLOAD["elev"]
    args, x = synthetic_swarm(N, deg)
    eng = gopt.BezOptimization(**args)._engine(True)
    J = eng.jac_separation(x, E, dense=False)
    torch.cuda.synchronize()
    res["c4_sep_sweep_checksum"] = checksum(J)
    res["c4_speed_sweep_checksum"] = checksum(eng.jac_speed(x, E, -1.0, dense=False))
    gb = J.numel() * 8 / 1e9
    ms = []
    for _ in range(3):                               # bursts of `reps` launches after an idle pause
        time.sleep(0.5)
        eng.jac_separation(x, E, dense=False, out=J)
        torch.cuda.synchronize()
        ms.append(timed(lambda: eng.jac_separation(x, E, dense=False, out=J), reps)[0])
    res["c4_sep_sweep_ms"] = ms
    res["c4_sep_sweep_gb"] = gb
    print("W2RESULT " + json.dumps(res), flush=True)


def w2(parent_root, rounds, reps, scratch):
    builds = {"this": ROOT}
    if parent_root:
        builds["parent"] = os.path.abspath(parent_root)
    runs = {k: [] for k in builds}
    dumps = {}
    for r in range(rounds):
        for k, root in builds.items():
            dump = os.path.join(scratch, k) if r == 0 else ""
            if dump:
                os.makedirs(dump, exist_ok=True)
                dumps[k] = dump
            code = ("import sys; sys.path.insert(0, %r); sys.path.insert(1, %r); import bench_batch_jac as t; "
                    "t.worker(%d, %r)" % (root, os.path.join(ROOT, "tools"), reps, dump))
            env = dict(os.environ, PYTHONPATH=root)
            p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, env=env)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("W2RESULT ")]
            if p.returncode != 0 or not line:
                raise RuntimeError("W2 worker (%s) failed:\n%s\n%s" % (k, p.stdout[-2000:], p.stderr[-4000:]))
            runs[k].append(json.loads(line[0][len("W2RESULT "):]))
            print(k, json.dumps(runs[k][-1]), flush=True)
    out = {}
    for k, rs in runs.items():
        ms = [v for rr in rs for v in rr["c4_sep_sweep_ms"]]
        out[k] = {"c4_sep_sweep_median_ms": float(np.median(ms)), "c4_sep_sweep_ms": ms,
                  "c4_sep_sweep_GBs": rs[0]["c4_sep_sweep_gb"] / (np.median(ms) * 1e-3),
                  "checksums": {c: sorted({rr[c] for rr in rs}) for c in ("c4_sep_sweep_checksum",
                                                                            "c4_speed_sweep_checksum")}}
    if "parent" in out:
        out["this_over_parent"] = out["this"]["c4_sep_sweep_median_ms"] / out["parent"]["c4_sep_sweep_median_ms"]
        same = {c: out["this"]["checksums"][c] == out["parent"]["checksums"][c] and len(out["this"]["checksums"][c]) == 1
                for c in ("c4_sep_sweep_checksum", "c4_speed_sweep_checksum")}
        for f in sorted(os.listdir(dumps["this"])):
            a, b = np.load(os.path.join(dumps["this"], f)), np.load(os.path.join(dumps["parent"], f))
            same[f[:-4]] = bool(a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64)))
        out["bit_identical_to_parent"] = same
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--w2-rounds", type=int, default=3)
    ap.add_argument("--parent-root", default=None,
                    help="checkout of the parent commit with its library built (W2 A/B and bit-identity)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_batch_jac.json"))
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    r1 = w1(a.M, a.rounds, a.reps)
    print(json.dumps(r1), flush=True)
    torch.cuda.empty_cache()
    with tempfile.TemporaryDirectory() as scratch:
        r2 = w2(a.parent_root, a.w2_rounds, 4, scratch)
    print(json.dumps(r2), flush=True)
    info_after = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"device": info, "device_after": info_after, "W1_c5_batch": r1, "W2_c4_single_point": r2}, f,
                  indent=1)


if __name__ == "__main__":
    main()
