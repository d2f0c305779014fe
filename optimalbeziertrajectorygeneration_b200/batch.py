"""Batches of independent trajectory problems (BASELINE.json configs[4], SURVEY 8(d) "C5").

The reference solves one problem per Python process; its SLSQP loop asks every
constraint callable for the base point and the nvar finite-difference points one after
the other (scipy/optimize/_slsqp_py.py:349-367 -> _numdiff.py:683-712).  Here M problems
that share the model (vehicles, degree, end conditions, bounds) and differ in their
point obstacles and in x are evaluated together: all M x (nvar+1) points of the M FD
sweeps go through the fused kernels in one launch per constraint block, and the
2-point quotients are formed on the device.  Problems are independent, so a multi-GPU
run deals them out in contiguous blocks (sharding.block_range) with no collective.

Only rows that depend on x are produced: the pairs that contain a vehicle (they are a
prefix of the lexicographic pair list because vehicles precede obstacles, Q8); the
obstacle-obstacle rows of the reference's vector are constants.
"""
import numpy as np
import torch

from . import optimization as _opt


class ProblemBatch:
    """``template`` = BezOptimization keyword arguments without ``pointObstacles``;
    ``obstacle_sets`` [M, nObs, dim] = the point obstacles of each problem."""

    def __init__(self, template, obstacle_sets, device=None):
        obstacle_sets = np.ascontiguousarray(obstacle_sets, dtype=np.float64)
        if obstacle_sets.ndim != 3:
            raise ValueError("obstacle_sets must be [M, nObs, dim]")
        self.M, self.nObs = int(obstacle_sets.shape[0]), int(obstacle_sets.shape[1])
        args = dict(template)
        args["pointObstacles"] = [list(o) for o in obstacle_sets[0]]
        self.bezopt = _opt.BezOptimization(**args)
        self.eng = self.bezopt._engine(with_obstacles=True)
        if device is not None and torch.device("cuda", device) != self.eng.device:
            raise ValueError("ProblemBatch lives on the current CUDA device")
        if obstacle_sets.shape[2] != self.eng.dim:
            raise ValueError("obstacles are %d-dimensional, the model is %d-dimensional"
                             % (obstacle_sets.shape[2], self.eng.dim))
        self.d_obst = torch.as_tensor(obstacle_sets, device=self.eng.device)
        self.nvar = self.eng.nvar
        N, nObs = self.eng.N, self.nObs
        self.npairs_x = N * (N - 1) // 2 - nObs * (nObs - 1) // 2     # pairs that contain a vehicle
        self.model = self.bezopt.model

    # ------------------------------------------------------------------
    def fd_points(self, X):
        """host X [M, nvar] -> device (Xp [M, nvar+1, nvar], dx [M, nvar]): the base point and the
        nvar forward points of every problem, h and dx as SciPy chooses them (ConstraintEngine.fd_points)."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        if X.shape != (self.M, self.nvar):
            raise ValueError("X must be [%d, %d]" % (self.M, self.nvar))
        return self.eng.fd_points(X)

    def evaluate(self, d_X, evals_per_problem, elev=None, blocks=("sep", "maxspeed", "angrate")):
        """d_X [M * evals_per_problem, nvar] (device) -> {block: [M * evals_per_problem, m_block]}.
        sep: the npairs_x x-dependent pairs x L; maxspeed: numVeh x L; angrate: numVeh x (4(n+E)+1)."""
        E = _opt._deg_elev() if elev is None else int(elev)
        cpts, tf = self.eng.assemble(d_X, E, obst_sets=self.d_obst, evals_per_set=int(evals_per_problem))
        return self._values(cpts, tf, E, blocks)

    def _values(self, cpts, tf, E, blocks):
        """The blocks of evaluate() at assembled points cpts [Q, N, S], tf [Q]."""
        eng, m = self.eng, self.model
        Q = int(cpts.shape[0])
        res = {}
        if "sep" in blocks:
            res["sep"] = eng.separation(cpts, E, m["maxSep"], pair_begin=0, npairs=self.npairs_x).view(Q, -1)
        if "maxspeed" in blocks:
            res["maxspeed"] = eng.speed(cpts, tf, E, -1.0, float(m["maxSpeed"]) ** 2).view(Q, -1)
        if "minspeed" in blocks:
            res["minspeed"] = eng.speed(cpts, tf, E, 1.0, -float(m["minSpeed"]) ** 2).view(Q, -1)
        if "angrate" in blocks:
            res["angrate"] = eng.angrate(cpts, tf, E, -1.0, float(m["maxAngRate"]) ** 2).view(Q, -1)
        return res

    def sweep(self, X, elev=None, blocks=("sep", "maxspeed", "angrate")):
        """One finite-difference sweep of every problem: returns {block: (f0 [M, m], JT [M, nvar, m])}
        on the device, JT[p, k] = (f(x_p + h_k e_k) - f(x_p)) / dx_k (SciPy's 2-point formula).
        "sep_closed", "maxspeed_closed", "minspeed_closed", "angrate_closed": the same blocks in closed
        form (ConstraintEngine.jac_separation / jac_speed / jac_angrate_closed), same shapes as the
        literal blocks; they share one assembly of the M base points and evaluate f0 there only."""
        closed = tuple(b for b in blocks if b in _CLOSED)
        literal = tuple(b for b in blocks if b not in _CLOSED)
        Xp, dx = self.fd_points(X)
        eng = self.eng
        out = {}
        if literal:
            nv1 = self.nvar + 1
            F = self.evaluate(Xp.view(self.M * nv1, self.nvar), nv1, elev, literal)
            for name, f in F.items():
                f = f.view(self.M, nv1, -1)
                out[name] = (f[:, 0], eng.fd_quotient(f, dx))
        if closed:
            E = _opt._deg_elev() if elev is None else int(elev)
            cpts, tf = eng.assemble(Xp[:, 0].contiguous(), E, obst_sets=self.d_obst, evals_per_set=1)
            f0 = self._values(cpts, tf, E, tuple(_CLOSED[b] for b in closed))
            base = (cpts, tf, dx, True)
            for name in closed:
                if name == "sep_closed":
                    JT = eng.jac_separation(None, E, npairs=self.npairs_x, base=base)
                elif name == "angrate_closed":
                    JT = eng.jac_angrate_closed(None, E, -1.0, base=base)
                else:
                    JT = eng.jac_speed(None, E, -1.0 if name == "maxspeed_closed" else 1.0, base=base)
                out[name] = (f0[_CLOSED[name]], JT)
        return out


# closed-form sweep block -> the literal block it reproduces
_CLOSED = {"sep_closed": "sep", "maxspeed_closed": "maxspeed", "minspeed_closed": "minspeed",
           "angrate_closed": "angrate"}
