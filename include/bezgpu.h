/*
 * bezgpu.h -- C ABI of libbezgpu.so: the B200 (sm_100a) implementation of the
 * Bezier constraint-evaluation hot path of
 * caslabuiowa/OptimalBezierTrajectoryGeneration.
 *
 * Every entry point is what a binding for the reference would call in place of
 * the cited reference code (paths relative to the upstream repository root).
 * Conventions
 *   - all pointers named d_* are DEVICE pointers owned by the caller (PyTorch
 *     tensors in the Python host layer); h_* are HOST pointers.  The library
 *     allocates only plan-resident constant tables.
 *   - every launch is asynchronous on the caller's stream (a cudaStream_t
 *     passed as void*; NULL = legacy default stream).
 *   - return value: 0 = OK, > 0 = a cudaError_t, < 0 = argument error
 *     (BEZ_E*).  bez_last_error() returns a thread-local description.
 *   - all arithmetic is IEEE fp64.  Geometry entry points (split, extrema,
 *     GJK, minDist, collCheck) are compiled without FMA contraction so that
 *     they reproduce the reference's numba/numpy rounding (SURVEY Q13).
 *
 * Control-point layout in HBM ("vehicle rows"):   cpts[b][v][S]
 *     b = evaluation point (base or finite-difference perturbed x)   0..B-1
 *     v = curve index (vehicles first, then point obstacles)         0..N-1
 *     S = dim*(n+1) rounded up to an even count (16-byte aligned rows); entry
 *         d*(n+1)+k is control point k of dimension d, the pad entry is 0.
 * A warp that walks over 32 consecutive pairs (i, j..j+31) reads one row
 * (broadcast) plus one contiguous 32*S*8-byte span with 128-bit loads.
 */
#ifndef BEZGPU_H
#define BEZGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEZ_OK            0
#define BEZ_EINVAL       (-1)   /* bad argument                        */
#define BEZ_ENOMEM       (-2)   /* host allocation failed              */
#define BEZ_EUNSUPPORTED (-3)   /* degree / dimension out of range     */

/* Degree limits (one place; INTEGRATION.md section 4 quotes these):
 *   plans and the fused constraint / objective kernels   n <= BEZ_MAX_DEGREE      = 16
 *   the fp64 tensor-path variants of those kernels        n <= BEZ_MAX_DEGREE_MMA  = 15, dim >= 2 (TMA-store
 *                                                         variant for L <= 128, column-tiled variant above;
 *                                                         other shapes run the DFMA kernels)
 *   closed-form Jacobian kernels                          n <= BEZ_MAX_DEGREE_JAC  = 12
 *   angular rate                                          n + elev <= 250 (tensor path and closed-form
 *                                                         Jacobian <= 127) */
#define BEZ_MAX_DEGREE      16
#define BEZ_MAX_DEGREE_MMA  15
#define BEZ_MAX_DEGREE_JAC  12
#define BEZ_MAX_GEOM_PTS  32    /* n+1 <= 32 for split/GJK/minDist      */

typedef struct bez_plan bez_plan;

const char *bez_last_error(void);
int bez_version(void);

/* ---- plan: device-resident constant tables for one (n, dim, elev) ------
 * Replaces the class-level caches BezierParams.elevationMatrixCache /
 * productMatrixCache (bezier.py:48-52) and the table builders
 * elevMatrix (bezier.py:1127-1147), prodMatrix (bezier.py:1151-1176).
 * The caller builds the tables ON THE HOST with scipy.special.binom exactly
 * as the reference does (SURVEY Q14) and passes them in:
 *   h_prodW [(n+1)*(n+1)]   W[i][j] = C(n,i)C(n,j)/C(2n,i+j)
 *   h_elevT [(2n+1)*L]      T[j][i] = C(2n,j)C(E,i-j)/C(2n+E,i),  L = 2n+E+1
 *   h_elev1 [n*(n+1)]       elevMatrix(n-1,1) used by Bezier.diff (bezier.py:519)
 */
int bez_plan_create(int n, int dim, int elev, int device,
                    const double *h_prodW, const double *h_elevT,
                    const double *h_elev1, bez_plan **out);
int bez_plan_destroy(bez_plan *plan);
int bez_plan_info(const bez_plan *plan, int *n, int *dim, int *elev, int *L);

/* ---- A0: BezOptimization.reshapeVector (optimization.py:242-285) + the
 * point-obstacle stacking of temporalSeparationConstraints
 * (optimization.py:86-94), for B optimisation vectors at once.
 *   d_x        [B][nvar]
 *   fixed_ends 0/1 : initPoints/finalPoints given (columns 0 and n fixed)
 *   dubins     0/1 : initSpeeds given (columns 1 and n-1 from speed*tf/n*(cos,sin); dim must be 2)
 *   timeopt    0/1 : tf = x[nvar-1] else tf_fixed
 *   d_init/d_final [numVeh][dim]; d_ispeed/d_fspeed/d_icos/d_isin/d_fcos/d_fsin [numVeh]
 *   d_obst     [nObs][dim] (may be NULL when nObs == 0)
 *   d_cpts     [B][numVeh+nObs][S]          (output)
 *   d_tf       [B]                          (output; the tf each x implies)
 */
int bez_assemble_cpts(const bez_plan *plan, const double *d_x, int B, int nvar,
                      int numVeh, int nObs, int fixed_ends, int dubins, int timeopt,
                      double tf_fixed,
                      const double *d_init, const double *d_final,
                      const double *d_ispeed, const double *d_fspeed,
                      const double *d_icos, const double *d_isin,
                      const double *d_fcos, const double *d_fsin,
                      const double *d_obst,
                      double *d_cpts, double *d_tf, void *stream);
/* The same for a batch of independent problems that share the model and differ in their
 * point obstacles (BASELINE.json configs[4]: 65 536 Dubins problems x 16 obstacles x the
 * nvar+1 points of each problem's FD sweep):  d_obst is [nsets][nObs][dim] and evaluation
 * b takes set b / evals_per_obst_set (0 = one set for all, i.e. bez_assemble_cpts). */
int bez_assemble_cpts_sets(const bez_plan *plan, const double *d_x, int B, int nvar,
                           int numVeh, int nObs, int fixed_ends, int dubins, int timeopt,
                           double tf_fixed,
                           const double *d_init, const double *d_final,
                           const double *d_ispeed, const double *d_fspeed,
                           const double *d_icos, const double *d_isin,
                           const double *d_fcos, const double *d_fsin,
                           const double *d_obst, int evals_per_obst_set,
                           double *d_cpts, double *d_tf, void *stream);

/* ---- A1-A4: _temporalSeparationConstraints (optimization.py:311-346) =
 * Bezier.sub (bezier.py:347-374) -> normSquare/_normSquare (bezier.py:869-889,
 * 1724-1756; incl. the dim/2 factor, SURVEY Q1) -> elev(E) (bezier.py:469-495)
 * -> minus maxSep^2, fused, for the pairs [pair_begin, pair_begin+npairs) of
 * the lexicographic i<j list over N curves, for B evaluation points.
 *   d_out     [B][npairs][L]
 *   d_pairmin [B][npairs] or NULL: min over the L values of each pair (the
 *             quantity whose sign is the active-pair flag).
 */
int bez_pair_sepsq_elev(const bez_plan *plan, const double *d_cpts, int B, int N,
                        int64_t pair_begin, int64_t npairs, double maxSep2,
                        double *d_out, double *d_pairmin, void *stream);
/* The same kernel fused with the one collective of the path (SURVEY 8(e): all-gather of
 * the per-pair minima): every minimum is stored to d_pairmin AND, from inside the kernel,
 * to npeers <= BEZ_MAX_PEERS peer-GPU buffers over NVLink (h_peer_min: host array of
 * device pointers into the peers' gathered [world*B][npairs] matrices, each already offset
 * to this rank's block; peer access / symmetric memory is set up by the caller).  The
 * data is complete on a peer once this kernel has finished on every rank (stream-ordered
 * barrier by the caller).  BEZ_EUNSUPPORTED for shapes outside the tensor-path kernels. */
int bez_pair_sepsq_elev_p2p(const bez_plan *plan, const double *d_cpts, int B, int N,
                            int64_t pair_begin, int64_t npairs, double maxSep2,
                            double *d_out, double *d_pairmin,
                            const uint64_t *h_peer_min, int npeers, void *stream);

/* Reduced results of the two fused kernels (all device pointers, all optional; NULL = not
 * produced).  An "item" is a pair (bez_pair_sepsq_elev_ex) or a vehicle (bez_speed_sq_elev_ex);
 * f = b * nitems + item is its flattened index in the launch.  The quantity reduced is the
 * minimum over the item's L elevated values -- what Examples/SequentialSwarm.py:62-67 takes
 * (`.cpts.min()`) and whose sign is the active-constraint flag (SURVEY 8(c)).
 *   itemmin     [B][min_pitch] minima (min_pitch = 0 means nitems; a larger pitch lets ranks
 *               that own pair sub-ranges write into one [B][P] matrix)
 *   peer_min    host array of npeers <= BEZ_MAX_PEERS device addresses: the same matrix on
 *               other GPUs (NVLink peer / symmetric memory), each already offset like itemmin;
 *               every minimum is also stored there from inside the kernel (fused all-gather)
 *   active_mask bit (f & 31) of word f >> 5 is set iff min < threshold; ceil(B*nitems/32) words
 *   list_*      compacted list of the items with min < threshold: *list_count (zeroed by the
 *               caller) receives their number; entry k < list_cap holds list_idx[k] = f and
 *               list_val[k] = min (order unspecified; entries beyond list_cap are dropped but
 *               counted, so list_count > list_cap reports the overflow)
 * With d_out == NULL the pair kernel writes no rows at all (minima only). */
#define BEZ_MAX_PEERS 7
typedef struct bez_reduce_opts {
    double *itemmin;
    int64_t min_pitch;
    const uint64_t *peer_min;
    int npeers;
    uint32_t *active_mask;
    double threshold;
    uint64_t *list_count;
    int64_t *list_idx;
    double *list_val;
    int64_t list_cap;
} bez_reduce_opts;
int bez_pair_sepsq_elev_ex(const bez_plan *plan, const double *d_cpts, int B, int N,
                           int64_t pair_begin, int64_t npairs, double maxSep2,
                           double *d_out, const bez_reduce_opts *opts, void *stream);
int bez_speed_sq_elev_ex(const bez_plan *plan, const double *d_cpts, const double *d_tf,
                         int B, int N, int veh_begin, int nveh, double alpha, double beta,
                         double *d_out, const bez_reduce_opts *opts, void *stream);

/* ---- A5: _maxSpeedConstraints / _minSpeedConstraints (optimization.py:349-422)
 * = Bezier.diff (bezier.py:497-519, same degree, SURVEY Q3) -> normSquare ->
 * elev(E) -> alpha*value + beta, for vehicles [veh_begin, veh_begin+nveh).
 *   max speed: alpha=-1, beta=maxSpeed^2 ; min speed: alpha=+1, beta=-minSpeed^2
 *   d_tf  [B]      d_out [B][nveh][L]
 */
int bez_speed_sq_elev(const bez_plan *plan, const double *d_cpts, const double *d_tf,
                      int B, int N, int veh_begin, int nveh,
                      double alpha, double beta, double *d_out, void *stream);

/* ---- A6: _maxAngularRateConstraints -> _angularRateSqr (optimization.py:425-459,
 * 578-611) with Bezier.mul / multiplyBezCurves (bezier.py:376-432, 1211-1246):
 * 2-D vehicles only (the reference raises ValueError otherwise, optimization.py:590).
 * Tables (host, scipy.special.binom, m = n + elev):
 *   h_Tpos   [(n+1)*(m+1)]  elevMatrix(n, elev)
 *   h_elev1m [m*(m+1)]      elevMatrix(m-1, 1)
 *   h_Cm [m+1] = C(m,.)     h_C2m [2m+1] = C(2m,.)
 *   d_out [B][nveh][4m+1] = alpha * (num^2/den^2) + beta   (max rate: alpha=-1, beta=maxAngRate^2)
 *   row_stride = S of the control-point rows (see top of file)
 * m <= 250 (bez_angrate_tables_create refuses more).  The result does not depend on the spatial
 * unit: control points x 2^k give bit-identical outputs as long as the Bernstein coefficients of
 * num^2 and den^2 stay within about 1e+-150 (any m <= 250).
 */
typedef struct bez_angrate_tables bez_angrate_tables;
int bez_angrate_tables_create(int n, int elev, int device, const double *h_Tpos,
                              const double *h_elev1m, const double *h_Cm, const double *h_C2m,
                              bez_angrate_tables **out);
int bez_angrate_tables_destroy(bez_angrate_tables *tables);
int bez_angrate_sq(const bez_angrate_tables *tables, const double *d_cpts, const double *d_tf,
                   int B, int N, int row_stride, int veh_begin, int nveh,
                   double alpha, double beta, double *d_out, void *stream);

/* ---- A7: the finite-difference Jacobian SciPy's SLSQP forms from nvar+1 calls
 * of the constraint callables (scipy/optimize/_slsqp_py.py:349-367 ->
 * _numdiff.py:585-596, 683-712):  J[:,k] = (f(x+h_k e_k) - f(x)) / dx_k,
 * dx_k = (x_k+h_k) - x_k.  Both constraints are quadratic in the control points,
 * which are affine in x, so the quotient is evaluated in closed form
 *      J[:,k] = elev( scale * B(2a + dx_k*delta, delta) ),  delta = d a / d x_k
 * (no cancellation; only rows that depend on x_k are touched).
 *   d_cpts [N][S]   control points of the base x (bez_assemble_cpts with B = 1)
 *   ncols, offset   free control points per row of x and index of the first one
 *   d_dx   [nvar]   SciPy's divisors
 *   d_dir  [N][S]   d(control points)/d x_kdir for a variable that moves every
 *                   curve (tf of time-optimal problems), kdir = its index or -1
 *   dense = 1: d_out is J^T [nvar][ld] (zero-filled here, ld >= rows of the block;
 *              row k holds column k of J, so stores stay coalesced)
 *   dense = 0: sweep layout, [numVeh*dim*ncols][N-1][L] (partner curves in
 *              ascending order, the vehicle itself skipped) followed, when
 *              kdir >= 0, by [P][L] for the kdir column.
 * These two are the B = 1 case of the batched entries below (all P pairs; the scalar tf for the
 * speed rows): the same argument checks and the same kernel choice.
 */
int bez_jac_sepsq_elev(const bez_plan *plan, const double *d_cpts, int N, int numVeh,
                       int ncols, int offset, const double *d_dx, const double *d_dir,
                       int kdir, int dense, double *d_out, int64_t ld, void *stream);
/* speed rows: alpha as in bez_speed_sq_elev; sweep layout [numVeh*dim*ncols][L]
 * (+ [numVeh][L] for kdir). */
int bez_jac_speed_sq_elev(const bez_plan *plan, const double *d_cpts, int N, int numVeh,
                          int ncols, int offset, double tf, double alpha,
                          const double *d_dx, const double *d_dir, int kdir, int dense,
                          double *d_out, int64_t ld, void *stream);

/* The same two Jacobians at B base points at once (problem batches, multi-start points): point b
 * has its own control points, divisors, tf and output block; the direction rows are shared.
 *   d_cpts [B][N][S]  base points (bez_assemble_cpts / bez_assemble_cpts_sets)
 *   d_dx   [B][nvar]  nvar = numVeh*dim*ncols (+ 1 with kdir >= 0)
 *   kdir   -1, or numVeh*dim*ncols for the tf variable of time-optimal models; d_dir may then be
 *          NULL: tf moves no control point (its separation rows are zero, its speed rows carry
 *          only the n/tf factor)
 *   npairs the leading pairs of the lexicographic list that get rows: at least every pair that
 *          contains a vehicle (P - nObs(nObs-1)/2, vehicles precede obstacles), at most P
 *   d_tf   [B] tf of each point (the tf that bez_assemble_cpts returned)
 *   dense = 1: d_out is J^T [B][nvar][ld], ld >= npairs*L (separation) or numVeh*L (speed);
 *              entries no item writes (pairs without the variable's vehicle) are zero-filled
 *   dense = 0: separation [B][numVeh*dim*ncols*(N-1) + (kdir >= 0 ? npairs : 0)][L],
 *              speed [B][numVeh*dim*ncols + (kdir >= 0 ? numVeh : 0)][L]; ld is ignored
 * With one vehicle (and npairs = N-1, ld = the block), a point's dense block is its sweep block,
 * and a dense request runs as a sweep.
 * B = 0 is a no-op.  BEZ_EINVAL for NULL pointers, negative sizes, a kdir other than -1 or
 * numVeh*dim*ncols, npairs or ld out of range; BEZ_EUNSUPPORTED above BEZ_MAX_DEGREE_JAC.
 * Arguments are checked before any CUDA call. */
int bez_jac_sepsq_elev_batched(const bez_plan *plan, const double *d_cpts, int B, int N,
                               int numVeh, int ncols, int offset, const double *d_dx,
                               const double *d_dir, int kdir, int64_t npairs, int dense,
                               double *d_out, int64_t ld, void *stream);
int bez_jac_speed_sq_elev_batched(const bez_plan *plan, const double *d_cpts, const double *d_tf,
                                  int B, int N, int numVeh, int ncols, int offset, double alpha,
                                  const double *d_dx, const double *d_dir, int kdir, int dense,
                                  double *d_out, int64_t ld, void *stream);

/* Literal 2-point quotient (scipy/optimize/_numdiff.py:709-711) for constraint
 * blocks without a closed form (angular rate): d_F [nvar+1][m] holds f(x0) in row
 * 0 and f(x0 + h_k e_k) in row k+1; d_JT [nvar][m] = (F[k+1] - F[0]) / dx[k]
 * (bez_fd_quotient_batched with count = 1). */
int bez_fd_quotient(const double *d_F, const double *d_dx, int nvar, int64_t m,
                    double *d_JT, void *stream);
/* count independent sweeps: d_F [count][nvar+1][m], d_dx [count][nvar], d_JT [count][nvar][m] */
int bez_fd_quotient_batched(const double *d_F, const double *d_dx, int64_t count, int nvar,
                            int64_t m, double *d_JT, void *stream);

/* Closed-form 2-point quotient of the angular-rate block (bez_angrate_sq with alpha, any beta):
 * the block is a control-point-wise ratio QQ / SS of two Bernstein squares of bilinear forms in the
 * control points, and P(a', a') - P(a, a) = P(a' - a, a' + a) (P = Bernstein product) gives every
 * difference without cancellation (DESIGN section 3.3).  Matches the exactly rounded quotient, and
 * writes only the rows of the vehicle a control-point variable moves.  n + elev <= 127
 * (BEZ_EUNSUPPORTED above: bez_fd_quotient covers those shapes).
 *   d_cpts  [B][N][row_stride]  base points (vehicles 0..numVeh-1 are used);  d_tf [B]
 *   nvar    numVeh*2*ncols (+ 1 with kdir >= 0); variables in x's order (vehicle, dimension,
 *           free column; control point = column + offset), then tf
 *   d_dx    [B][nvar] SciPy's divisors
 *   d_dir   [N][row_stride] d(control points)/d tf, or NULL (tf moves no control point)
 *   kdir    nvar-1 for time-optimal models (tf also scales the derivatives), else -1
 *   dense = 1: d_out is J^T [B][nvar][ld], zero-filled here, ld >= numVeh*(4m+1)
 *   dense = 0: [B][numVeh*2*ncols + (kdir >= 0 ? numVeh : 0)][4m+1]: one row per control-point
 *              variable in x's order, then one tf row per vehicle
 *   d_scratch bez_jac_angrate_scratch_doubles(B, numVeh, n, elev) doubles:
 *              B*numVeh*(128*U + 432), U = ceil((n+elev+1)/8); 0 for unsupported shapes */
size_t bez_jac_angrate_scratch_doubles(int B, int numVeh, int n, int elev);
int bez_jac_angrate_sq(const bez_angrate_tables *tables, const double *d_cpts, const double *d_tf,
                       int B, int N, int row_stride, int numVeh, int ncols, int offset, int nvar,
                       const double *d_dx, const double *d_dir, int kdir, double alpha, int dense,
                       double *d_scratch, double *d_out, int64_t ld, void *stream);

/* ---- single-curve algebra behind the bezier.Bezier methods, batched over
 * independent rows/curves; tables are DEVICE arrays the caller built on the host
 * with scipy.special.binom (same expressions as the reference, SURVEY Q14).
 *   bez_curve_elev   Bezier.elev        bezier.py:469-495   d_T = elevMatrix(n,R) [n+1][n+R+1]
 *   bez_curve_diff   Bezier.diff        bezier.py:497-519   d_E1 = elevMatrix(n-1,1); d_T[rows/rows_per_T] = tf-t0
 *   bez_curve_mul    Bezier.mul         bezier.py:376-432   d_W [m+1][n+1] = C(m,i)C(n,j)/C(m+n,i+j)
 *   bez_curve_normsq Bezier.normSquare  bezier.py:869-889   d_cpts [curves][dim][n+1] -> [curves][2n+1] (x dim/2, Q1)
 *   bez_curve_eval   Bezier.__call__/.curve -> deCasteljauCurve bezier.py:944-982 (bit exact, no FMA)
 */
int bez_curve_elev(const double *d_cpts, const double *d_T, int64_t rows, int n, int R,
                   double *d_out, void *stream);
int bez_curve_diff(const double *d_cpts, const double *d_E1, const double *d_T, int64_t rows,
                   int64_t rows_per_T, int n, double *d_out, void *stream);
int bez_curve_mul(const double *d_a, const double *d_b, const double *d_W, int64_t rows, int m, int n,
                  double *d_out, void *stream);
int bez_curve_normsq(const double *d_cpts, const double *d_W, int64_t curves, int dim, int n,
                     double *d_out, void *stream);
int bez_curve_eval(const double *d_cpts, const double *d_tau, int64_t rows, int n, int ntau,
                   double t0, double tf, double *d_out, void *stream);

/* ---- A14: cost callables (optimization.py:287-308, 462-519) on assembled control
 * points d_cpts [B][N][S]; d_out [B].  euclidean = total control-polygon length
 * (_euclideanObjective; for dim 2 the reference reads an uninitialised third
 * component, SURVEY Q10 -- here it is 0); accel = sum of the control points of
 * elev(normSquare(diff(diff(pos))), E) over the vehicles (_minAccelObjective). */
int bez_objective_euclidean(const bez_plan *plan, const double *d_cpts, int B, int N, int numVeh,
                            double *d_out, void *stream);
int bez_objective_accel(const bez_plan *plan, const double *d_cpts, const double *d_tf, int B,
                        int N, int numVeh, double *d_out, void *stream);

/* Gradient of the cost callables as SciPy forms it for SLSQP ('2-point' rule on
 * objectiveFunction, scipy/optimize/_slsqp_py.py:424-426 -> _numdiff.py:585-596, 683-712):
 * d_out[k] = (f(x + dx_k e_k) - f(x)) / dx_k for the numVeh*dim*ncols control-point variables
 * (row-major (vehicle, dimension, free column); free column col = control point col + offset,
 * optimization.py:242-285), in cancellation-free closed form from the assembled control points
 * d_cpts [N][S] of the base x.  kind 0 = euclidean (optimization.py:462-489), 1 = accel
 * (optimization.py:503-519, tf = the model's tf).  Replaces nvar+1 host calls of the callable. */
int bez_objective_grad(const bez_plan *plan, const double *d_cpts, int kind, double tf, int numVeh,
                       int ncols, int offset, const double *d_dx, double *d_out, void *stream);

/* ---- A8: Bezier.split -> deCasteljauSplit (bezier.py:533-572, 985-1027), bit exact.
 *   d_cpts [count][dim][n+1]; d_tlocal [count] = (tDiv - t0)/(tf - t0); outputs same shape,
 *   right half already in ascending order (bezier.py:563).  One warp per curve. */
int bez_split(const double *d_cpts, const double *d_tlocal, int count, int dim, int n,
              double *d_left, double *d_right, void *stream);

/* ---- A9: Bezier.min / Bezier.max (bezier.py:631-667, 727-763), the intended
 * algorithm (split at the extreme control point's local parameter; the reference
 * extrapolates beyond depth 1, SURVEY Q4).  d_rows [count][n+1]; d_status 1 = depth limit.
 * d_scratch: bez_extrema_scratch_doubles(count, n, max_depth) doubles. */
size_t bez_extrema_scratch_doubles(int count, int n, int max_depth);
int bez_extrema(const double *d_rows, int count, int n, double tol, int maximum, int max_depth,
                double *d_scratch, double *d_out, int *d_status, void *stream);

/* ---- A10: gjkNew (gjk/gjk.py:229-360 and helpers :87-114, :397-477, :493-681).
 *   d_poly1 [count][n1max][3], d_n1 [count] or NULL (= n1max each); likewise poly2.
 *   d_flag: 1 distance available / 0 collision / -1 iteration limit;
 *   d_p1, d_p2 [count][3], d_dist [count] (NaN unless flag == 1).  One warp per pair. */
int bez_gjk(const double *d_poly1, const double *d_poly2, const int *d_n1, const int *d_n2,
            int n1max, int n2max, int count, int *d_flag, double *d_p1, double *d_p2,
            double *d_dist, void *stream);

/* ---- A11: Bezier.minDist -> _minDist (bezier.py:840-852, 1283-1408, 1499-1516).
 *   d_c1 [count][dim1][n1+1], d_c2 [count][dim2][n2+1] (2-D curves are z-padded);
 *   d_out [count][3] = (alpha, t1, t2), NaN when d_status != 0; status bit 1 = a path
 *   reached max_depth (the reference raises RecursionError there, SURVEY Q6: the search
 *   is aborted), bit 4 = more than max_nodes GJK calls. */
size_t bez_mindist_scratch_doubles(int count, int n1, int n2, int max_depth);
int bez_mindist(const double *d_c1, const double *d_c2, int count, int dim1, int dim2, int n1,
                int n2, double eps, int max_depth, long long max_nodes, double *d_scratch,
                double *d_out, int *d_status, void *stream);

/* ---- A12: minDist2Poly / collCheck / collCheck2Poly (bezier.py:1411-1496,
 * 1535-1547, 1561-1651).  d_polys [count][mmax][3], d_npoly [count] or NULL.
 *   mindist2poly d_out [count][5] = (alpha, t1, closest point xyz); status bit 1 =
 *     depth limit, bit 2 = no closest point (the reference returns -1 there).
 *   collcheck    d_out [count] = 1 (separated) / alpha (0.0 = contact) / -1 (depth 100)
 *   collcheck2poly d_out [count] = 1 / 0; d_status 1 = node budget exhausted. */
size_t bez_mindist2poly_scratch_doubles(int count, int n1, int max_depth);
int bez_mindist2poly(const double *d_c1, const double *d_polys, const int *d_npoly, int count,
                     int dim1, int n1, int mmax, double eps, int max_depth, long long max_nodes,
                     double *d_scratch, double *d_out, int *d_status, void *stream);
size_t bez_collcheck_scratch_doubles(int count, int n1, int n2);
int bez_collcheck(const double *d_c1, const double *d_c2, int count, int dim1, int dim2, int n1,
                  int n2, double eps, double *d_scratch, double *d_out, void *stream);
size_t bez_collcheck2poly_scratch_doubles(int count, int n1);
int bez_collcheck2poly(const double *d_c1, const double *d_polys, const int *d_npoly, int count,
                       int dim1, int n1, int mmax, long long max_nodes, double *d_scratch,
                       double *d_out, int *d_status, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BEZGPU_H */
