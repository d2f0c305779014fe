// Finite-difference Jacobian columns of the separation and speed constraints
// (A7 of SURVEY.md section 8) for sm_100a.
//
// SciPy's SLSQP forms  J[:,k] = (f(x + h_k e_k) - f(x)) / dx_k,  dx_k = (x_k+h_k) - x_k
// with nvar+1 calls of the constraint callable (scipy/optimize/_slsqp_py.py:349-367,
// _numdiff.py:585-596, 683-712).  Both constraints are quadratic forms of the control
// points, which are affine in x (reshapeVector), so the quotient has the closed form
//     J[:,k] = elev( scale * B(2a + dx*delta, delta) )
// where a is the curve being squared (c_i - c_j, or the derivative curve), delta =
// d a / d x_k and B is the Bernstein product.  Evaluating that directly is free of the
// cancellation that limits the literal difference to ~1e-7 relative accuracy, costs the
// same fused "square -> fold -> elevate" pipeline as one constraint row, and only
// touches the rows that depend on x_k:
//   J_PAIR_VAR   item = (variable kk of vehicle v, partner u != v)     N-1 rows per variable
//   J_PAIR_DIR   item = pair p, for a variable that moves every curve (tf of time-optimal
//                Dubins problems): delta = dir_i - dir_j, dir = d y / d tf
//   J_SPEED_VAR  item = variable kk -> the speed row of its vehicle
//   J_SPEED_DIR  item = vehicle v, tf variable (moves control points and the n/tf factor)
// Output either in the sweep layout [item][L] or scattered into a dense J^T [nvar][ld]
// (rows of J^T are contiguous, so stores stay coalesced; the host hands SciPy J^T.T).
//
// Batches of B base points (problem batches, multi-start): every mode's items repeat per point b,
// each with its own control points, divisors, tf and output block; the direction rows are shared.
// Work is cut into 32-item tiles per point (tile w -> point w / tiles_per_point), so a tile never
// straddles two points: its rows stay one contiguous run of the point's output block even where the
// point's direction rows sit between its variable rows and the next point's, and the tensor-path
// tile store and the partner-row runs of the TMA fetch apply unchanged.
#include <stdlib.h>

#include "sq_elev_core.cuh"
#include "sq_elev_mma.cuh"
#include "sq_elev_ws.cuh"

namespace {
using namespace bezcore;

enum JMode { J_PAIR_VAR = 0, J_PAIR_DIR = 1, J_SPEED_VAR = 2, J_SPEED_DIR = 3 };

template <int N_>
struct FullWeights { double w[(N_ + 1) * (N_ + 1)]; };

struct JacArgs {
    int early_store;      // A/B: proxy fence + bulk store right behind each m-tile (BEZGPU_MMA_FLAGS bit 8)
    const double *cpts;   // [B][N][S] base points
    const double *dir;    // [N][S] d y / d x_kdir (DIR modes; shared by all points)
    const double *dx;     // [B][nvar]
    const double *tfs;    // [B] tf of each point (SPEED modes), or NULL: the scalar tf
    const double *PQ;     // folded elevation table
    double *out;
    long long nitems;     // items per point
    long long tpp;        // 32-item tiles per point
    long long B;
    long long cstride, dxstride, ostride;   // doubles between consecutive points' cpts, dx, output
    long long ld;         // dense: row length of J^T
    int N, numVeh, L, Lh, LhPad;
    int ncols, offset;    // free columns per row of x, first free control point
    int kdir;             // variable index served by the DIR modes
    int dense;
    double tf;            // SPEED modes
    double scale;         // alpha * dim / 2
};

// Stage 1 of the Jacobian kernels for one item: s = B(2a + dx*delta, delta) (unscaled) and
// the offset of the item's output row.
// J_PAIR_VAR item = (variable kk, partner curve u): owner vehicle v, dimension d, control point c
struct PairVarItem { long long kk; int v, d, c, u; };
__device__ __forceinline__ PairVarItem pair_var_item(const JacArgs &A, int dim, long long item) {
    PairVarItem it;
    const int dim_ncols = dim * A.ncols;
    it.kk = item / (A.N - 1);
    const int uu = (int)(item - it.kk * (A.N - 1));
    it.v = (int)(it.kk / dim_ncols);
    const int rem = (int)(it.kk - (long long)it.v * dim_ncols);
    it.d = rem / A.ncols;
    it.c = A.offset + (rem - it.d * A.ncols);
    it.u = uu + (uu >= it.v ? 1 : 0);
    return it;
}

// Tile w of the flattened [B][tpp] tile list: point b, first item t0 of the point, live lanes cnt.
struct JacTile { long long b, t0; int cnt; };
__device__ __forceinline__ JacTile jac_tile(const JacArgs &A, long long w) {
    JacTile t;
    t.b = A.B == 1 ? 0 : w / A.tpp;
    t.t0 = (w - t.b * A.tpp) << 5;
    t.cnt = (int)((A.nitems - t.t0) < 32 ? (A.nitems - t.t0) : 32);
    return t;
}

// urow (J_PAIR_VAR only, optional): the partner curve's whole row, already in shared memory.
// ONEHOT + scratch (J_PAIR_VAR only): 2n+1 doubles of shared memory private to the lane (may alias
// the urow region of the warp: every lane has read its row before anyone writes).  With it the
// Bernstein product uses that delta = +-e_c is one-hot: s[i + c] = w[i][c] * (u_i * sg) -- the same
// bits as the dense double loop (all its other terms add +-0), 22 instead of 242 fp64 instructions.
template <int N_, int DIM, int JMODE, bool ONEHOT = false>
__device__ __forceinline__ void jac_stage1(const JacArgs &A, const FullWeights<N_> &FW,
                                           const DiffWeights<N_> &DW, long long b, long long item,
                                           double (&s)[2 * N_ + 1], long long &ro, const double *urow = nullptr,
                                           double *scratch = nullptr) {
    constexpr int NC = N_ + 1;
    constexpr int S = (DIM * NC + 1) / 2 * 2;
    constexpr bool DIRMODE = (JMODE == J_PAIR_DIR || JMODE == J_SPEED_DIR);
    constexpr int ND = DIRMODE ? DIM : 1;
    const int dim_ncols = DIM * A.ncols;
    const double *cpts = A.cpts + b * A.cstride;     // this point's control points and divisors
    const double *dxs = A.dx + b * A.dxstride;
    double a[ND][NC], dl[ND][NC];
    double dxk;
    int c_hot = 0;              // J_PAIR_VAR: delta = sg_hot * e_{c_hot}
    double sg_hot = 0.0;
    if (JMODE == J_PAIR_VAR) {
        const PairVarItem it = pair_var_item(A, DIM, item);
        const long long kk = it.kk;
        const int v = it.v, d = it.d, c = it.c, u = it.u;
        const int vi = v < u ? v : u, vj = v < u ? u : v;
        const double sg = v < u ? 1.0 : -1.0;
        c_hot = c;
        sg_hot = sg;
        const double *pv = cpts + (size_t)v * S + d * NC;
        if (urow) {                                 // partner row from shared memory (TMA row fetch)
            const double *pu = urow + d * NC;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const double cv = __ldg(pv + k), cu = pu[k];
                a[0][k] = v < u ? cv - cu : cu - cv;
                dl[0][k] = (k == c) ? sg : 0.0;
            }
        } else {
            const double *pu = cpts + (size_t)u * S + d * NC;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const double cv = __ldg(pv + k), cu = __ldg(pu + k);
                a[0][k] = v < u ? cv - cu : cu - cv;
                dl[0][k] = (k == c) ? sg : 0.0;
            }
        }
        dxk = __ldg(dxs + kk);
        const long long p = bez_pair_row_offset(vi, A.N) + (vj - vi - 1);
        ro = b * A.ostride + (A.dense ? kk * A.ld + p * A.L : item * (long long)A.L);
    } else if (JMODE == J_PAIR_DIR) {
        int vi, vj;
        bez_pair_decode(item, A.N, vi, vj);
#pragma unroll
        for (int d = 0; d < DIM; ++d)
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                a[d][k] = __ldg(cpts + (size_t)vi * S + d * NC + k) -
                          __ldg(cpts + (size_t)vj * S + d * NC + k);
                dl[d][k] = __ldg(A.dir + (size_t)vi * S + d * NC + k) -
                           __ldg(A.dir + (size_t)vj * S + d * NC + k);
            }
        dxk = __ldg(dxs + A.kdir);
        ro = b * A.ostride + (A.dense ? (long long)A.kdir * A.ld + item * A.L : item * (long long)A.L);
    } else if (JMODE == J_SPEED_VAR) {
        const long long kk = item;
        const int v = (int)(kk / dim_ncols);
        const int rem = (int)(kk - (long long)v * dim_ncols);
        const int d = rem / A.ncols;
        const int c = A.offset + (rem - d * A.ncols);
        const double val = (double)N_ / (A.tfs ? __ldg(A.tfs + b) : A.tf);
        const double *pv = cpts + (size_t)v * S + d * NC;
        double pt[NC], dd[NC], de[NC];
#pragma unroll
        for (int k = 0; k < NC; ++k) pt[k] = __ldg(pv + k);
#pragma unroll
        for (int k = 0; k < N_; ++k) {
            dd[k] = pt[k] * (-val) + pt[k + 1] * val;
            de[k] = ((k == c) ? -val : 0.0) + ((k + 1 == c) ? val : 0.0);
        }
        dd[N_] = 0.0; de[N_] = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            double q = dd[k] * DW.lo[k], r = de[k] * DW.lo[k];
            if (k > 0) { q = dd[k - 1] * DW.hi[k] + q; r = de[k - 1] * DW.hi[k] + r; }
            a[0][k] = q;
            dl[0][k] = r;
        }
        dxk = __ldg(dxs + kk);
        ro = b * A.ostride + (A.dense ? kk * A.ld + (long long)v * A.L : item * (long long)A.L);
    } else {   // J_SPEED_DIR: tf moves the control points (dir) and the n/tf factor
        const int v = (int)item;
        dxk = __ldg(dxs + A.kdir);
        const double tf = A.tfs ? __ldg(A.tfs + b) : A.tf;
        const double val = (double)N_ / tf;
        const double valp = (double)N_ / (tf + dxk);
        const double gam = -(double)N_ / (tf * (tf + dxk));         // (valp - val) / dx
#pragma unroll
        for (int d = 0; d < DIM; ++d) {
            double pt[NC], pd[NC], dd[NC], de[NC];
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                pt[k] = __ldg(cpts + (size_t)v * S + d * NC + k);
                pd[k] = A.dir ? __ldg(A.dir + (size_t)v * S + d * NC + k) : 0.0;   // NULL: tf moves no point
            }
#pragma unroll
            for (int k = 0; k < N_; ++k) {
                dd[k] = pt[k] * (-val) + pt[k + 1] * val;
                de[k] = valp * (pd[k + 1] - pd[k]) + gam * (pt[k + 1] - pt[k]);
            }
            dd[N_] = 0.0; de[N_] = 0.0;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                double q = dd[k] * DW.lo[k], r = de[k] * DW.lo[k];
                if (k > 0) { q = dd[k - 1] * DW.hi[k] + q; r = de[k - 1] * DW.hi[k] + r; }
                a[d][k] = q;
                dl[d][k] = r;
            }
        }
        ro = b * A.ostride + (A.dense ? (long long)A.kdir * A.ld + (long long)v * A.L : item * (long long)A.L);
    }

    if (ONEHOT && JMODE == J_PAIR_VAR) {
        __syncwarp();
#pragma unroll
        for (int k = 0; k <= 2 * N_; ++k) scratch[k] = 0.0;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const double ui = fma(dxk, dl[0][i], 2.0 * a[0][i]);
            scratch[i + c_hot] = fma(FW.w[i * NC + c_hot], ui * sg_hot, 0.0);
        }
#pragma unroll
        for (int k = 0; k <= 2 * N_; ++k) s[k] = scratch[k];
        return;
    }
    // s = B(2a + dx*delta, delta)   (Bernstein product, full weight matrix)
#pragma unroll
    for (int k = 0; k <= 2 * N_; ++k) s[k] = 0.0;
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        double uvec[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) uvec[i] = fma(dxk, dl[d][i], 2.0 * a[d][i]);
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int j = 0; j < NC; ++j)
                s[i + j] = fma(FW.w[i * NC + j], uvec[i] * dl[d][j], s[i + j]);
    }
}

template <int N_, int DIM, int JMODE>
__global__ void __launch_bounds__(kThreads, 3)
jac_sq_elev_kernel(const JacArgs A, const FullWeights<N_> FW, const DiffWeights<N_> DW) {
    constexpr int NC = N_ + 1;
    constexpr int NT = 2 * N_ + 1;
    constexpr int RS = RowGeom<N_>::RS;
    constexpr int CPL = 2;
    extern __shared__ __align__(16) double smem[];
    // layout: [kWarps][32][RS] double2 rows | [NT][LhPad] table | [kWarps][32] row offsets
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double2 *rows = reinterpret_cast<double2 *>(smem) + (size_t)warp * 32 * RS;
    double *tab = smem + (size_t)kWarps * 32 * RS * 2;
    long long *rowoff = reinterpret_cast<long long *>(tab + (size_t)NT * A.LhPad) + warp * 32;

    for (int i = threadIdx.x; i < NT * A.LhPad; i += kThreads) tab[i] = __ldg(A.PQ + i);
    __syncthreads();

    const long long nwt = A.B * A.tpp;
    const long long gwarp = (long long)blockIdx.x * kWarps + warp;
    const long long nwarps = (long long)gridDim.x * kWarps;
    const int ngroups = (A.LhPad / 32 + CPL - 1) / CPL;

    for (long long wt = gwarp; wt < nwt; wt += nwarps) {
        const JacTile T = jac_tile(A, wt);
        const int cnt = T.cnt;
        {
            const long long item = T.t0 + (lane < cnt ? lane : cnt - 1);
            double s[2 * N_ + 1];
            long long ro;
            jac_stage1<N_, DIM, JMODE>(A, FW, DW, T.b, item, s, ro);
            rowoff[lane] = ro;
            double2 *row = rows + (size_t)lane * RS;
#pragma unroll
            for (int j = 0; j < N_; ++j) {
                const double lo = s[j] * A.scale, hi = s[2 * N_ - j] * A.scale;
                row[j] = make_double2(lo + hi, lo - hi);
            }
            row[N_] = make_double2(s[N_] * A.scale, 0.0);
        }
        __syncwarp();
        for (int g = 0; g < ngroups; ++g) {
            if (cnt == 32)
                sweep_columns<N_, CPL, false, true, true>(rows, tab, A.out, g, lane, 32, A.L, A.Lh, A.LhPad, 0.0, rowoff);
            else
                sweep_columns<N_, CPL, false, false, true>(rows, tab, A.out, g, lane, cnt, A.L, A.Lh, A.LhPad, 0.0, rowoff);
        }
        __syncwarp();
    }
}

// Sweep-layout variant on the fp64 tensor path (sq_elev_mma.cuh): the rows of consecutive
// items are contiguous, so the DMMA stage 2 + TMA bulk-store epilogue of the constraint
// kernels applies unchanged.  Used for the per-variable modes (one dimension live in stage 1).
template <int N_, int DIM, int JMODE>
__global__ void __launch_bounds__(kThreads, 2)
jac_sq_elev_mma_kernel(const JacArgs A, const FullWeights<N_> FW, const DiffWeights<N_> DW) {
    using namespace bezmma;
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t per_warp = (size_t)kRowsDoubles + 16 * (size_t)A.L;
    double *rows = smem + warp * per_warp;
    double *obuf = rows + kRowsDoubles;
    for (int i = lane; i < kRowsDoubles; i += 32) rows[i] = 0.0;     // padding slots must be 0
    const unsigned obuf_s = (unsigned)__cvta_generic_to_shared(obuf);
    BFrags<N_, 4> Bf;
    load_bfrags<N_, 4>(Bf, A.PQ, A.L, A.LhPad, lane);
    MinSinks no_sinks;
    memset(&no_sinks, 0, sizeof(no_sinks));
    __syncwarp();
    const long long nwt = A.B * A.tpp;
    const long long gwarp = (long long)blockIdx.x * kWarps + warp;
    const long long nwarps = (long long)gridDim.x * kWarps;
    for (long long wt = gwarp; wt < nwt; wt += nwarps) {
        const JacTile T = jac_tile(A, wt);
        const long long t0 = T.t0;
        const int cnt = T.cnt;
        double *pout = A.out + T.b * A.ostride;
        const bool base_aligned = (reinterpret_cast<uintptr_t>(pout) & 15u) == 0;
        {
            double s[2 * N_ + 1];
            long long ro;
            jac_stage1<N_, DIM, JMODE, JMODE == J_PAIR_VAR>(A, FW, DW, T.b, t0 + (lane < cnt ? lane : cnt - 1), s, ro,
                                                            nullptr, rows + lane * kRowStride);
            double *row = rows + lane * kRowStride;
#pragma unroll
            for (int j = 0; j < N_; ++j) {
                const double lo = s[j] * A.scale, hi = s[2 * N_ - j] * A.scale;
                row[slot_e(j)] = lo + hi;
                row[slot_o(j)] = lo - hi;
            }
            row[slot_e(N_)] = s[N_] * A.scale;
            if (JMODE == J_PAIR_VAR) {       // the scratch use of the row overwrote the padding slots of the k-steps
#pragma unroll
                for (int j = N_ + 1; j < 4 * Geom<N_>::KE; ++j) row[slot_e(j)] = 0.0;
#pragma unroll
                for (int j = N_; j < 4 * Geom<N_>::KO; ++j) row[slot_o(j)] = 0.0;
            }
        }
        __syncwarp();
        mma_tile<N_, 4, 0, true>(rows, obuf, obuf_s, Bf, pout + (size_t)t0 * A.L, no_sinks, t0, cnt, A.L, 0.0, lane,
                                 base_aligned, A.early_store != 0);
        __syncwarp();
    }
    if (lane == 0) bulk_wait_all();
}

// The same sweep kernel, warp-specialised like the pair kernel (sq_elev_ws.cuh): per scheduler one
// producer warp (stage 1 only) feeds two consumer warps (DMMA stage 2 + TMA bulk stores) through a
// ring of three row slots; no TMA row fetch here, the items of a tile read scattered rows.
template <int N_, int DIM, int JMODE>
__global__ void __launch_bounds__(bezws::kWsThreads, 1)
jac_sq_elev_ws_kernel(const JacArgs A, const FullWeights<N_> FW, const DiffWeights<N_> DW) {
    using namespace bezmma;
    using namespace bezws;
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int group = warp & 3;
    constexpr bool TMAROWS = (JMODE == J_PAIR_VAR);
    constexpr int S_ = (DIM * (N_ + 1) + 1) / 2 * 2;
    constexpr int kSlotD = TMAROWS ? slot_doubles<N_, DIM>() : kRowsDoubles;
    double *slots = smem + (size_t)group * kSlots * kSlotD;
    double *stag0 = smem + (size_t)4 * kSlots * kSlotD;
    const size_t stag_per = 16 * (size_t)A.L;
    const unsigned bars_s = (unsigned)__cvta_generic_to_shared(stag0 + kConsumers * stag_per) + 8u * kBarsPerGroup * group;
    auto full_b = [&](int s) { return bars_s + 8u * s; };
    auto empty_b = [&](int s) { return bars_s + 8u * (kSlots + s); };
    auto rows_b = [&](int s) { return bars_s + 8u * (2 * kSlots + s); };
    if (warp < kProducers) {
        for (int i = lane; i < kSlots * kSlotD; i += 32) slots[i] = 0.0;           // padding slots must be 0
        if (lane == 0) {
            for (int s = 0; s < kSlots; ++s) { mbar_init(full_b(s), 32); mbar_init(empty_b(s), 32); mbar_init(rows_b(s), 1); }
            mbar_fence_init();
        }
    }
    __syncthreads();
    const long long nwt = A.B * A.tpp;
    const long long ngroups = (long long)gridDim.x * 4, gidx = (long long)blockIdx.x * 4 + group;
    const long long t_begin = gidx * nwt / ngroups;
    const int n = (int)((gidx + 1) * nwt / ngroups - t_begin);
    if (warp < kProducers) {
        reg_dec<120>();
        for (int k = 0; k < n; ++k) {
            const int s = k % kSlots, use = k / kSlots;
            const JacTile T = jac_tile(A, t_begin + k);
            const int cnt = T.cnt;
            const double *cpts = A.cpts + T.b * A.cstride;
            double sc[2 * N_ + 1];
            long long ro;
            const long long item = T.t0 + (lane < cnt ? lane : cnt - 1);
            double *slot = slots + (size_t)s * kSlotD;
            if (TMAROWS) {
                // the partner rows of a tile are consecutive rows of the control-point array (one run
                // per variable, broken once at the owner vehicle): one TMA bulk copy per run
                const PairVarItem it = pair_var_item(A, DIM, item);
                // the owner's row and the step length go to L1 while the slot is awaited and the rows fly
                asm volatile("prefetch.global.L1 [%0];" :: "l"(cpts + (size_t)it.v * S_ + it.d * (N_ + 1)));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(cpts + (size_t)it.v * S_ + it.d * (N_ + 1) + N_));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(A.dx + T.b * A.dxstride + it.kk));
                if (use > 0) mbar_wait(empty_b(s), (unsigned)(use - 1) & 1u);
                const int pu = __shfl_up_sync(0xffffffffu, it.u, 1);
                const bool start = lane == 0 || it.u != pu + 1;
                const unsigned runs = __ballot_sync(0xffffffffu, start);
                const unsigned slot_s = (unsigned)__cvta_generic_to_shared(slot);
                fence_async_smem();
                if (lane == 0) mbar_arrive_expect_tx(rows_b(s), 32u * S_ * 8u);
                __syncwarp();
                if (start) {
                    const unsigned higher = lane == 31 ? 0u : (runs & (0xffffffffu << (lane + 1)));
                    const int end = higher ? __ffs(higher) - 1 : 32;
                    // a run never leaves the point's array: rows u .. u + len - 1 <= N - 1 (a tile holds items
                    // of one point only; dead lanes repeat the last item)
                    bulk_load(slot_s + (unsigned)lane * (S_ * 8u), cpts + (size_t)it.u * S_,
                              (unsigned)(end - lane) * (S_ * 8u), rows_b(s));
                }
                mbar_wait(rows_b(s), (unsigned)use & 1u);
                jac_stage1<N_, DIM, JMODE, true>(A, FW, DW, T.b, item, sc, ro, slot + lane * S_, slot + lane * kRowStride);
                __syncwarp();
            } else {
                jac_stage1<N_, DIM, JMODE>(A, FW, DW, T.b, item, sc, ro);
                if (use > 0) mbar_wait(empty_b(s), (unsigned)(use - 1) & 1u);
            }
            double *row = slot + lane * kRowStride;
#pragma unroll
            for (int j = 0; j < N_; ++j) {
                const double lo = sc[j] * A.scale, hi = sc[2 * N_ - j] * A.scale;
                row[slot_e(j)] = lo + hi;
                row[slot_o(j)] = lo - hi;
            }
            row[slot_e(N_)] = sc[N_] * A.scale;
            if (TMAROWS) {
#pragma unroll
                for (int j = N_ + 1; j < 4 * Geom<N_>::KE; ++j) row[slot_e(j)] = 0.0;
#pragma unroll
                for (int j = N_; j < 4 * Geom<N_>::KO; ++j) row[slot_o(j)] = 0.0;
            }
            mbar_arrive(full_b(s));
        }
    } else {
        reg_inc<192>();
        const int cidx = warp - kProducers, ci = cidx >> 2;
        double *obuf = stag0 + (size_t)cidx * stag_per;
        const unsigned obuf_s = (unsigned)__cvta_generic_to_shared(obuf);
        BFrags<N_, 4> Bf;
        load_bfrags<N_, 4>(Bf, A.PQ, A.L, A.LhPad, lane);
        MinSinks no_sinks;
        memset(&no_sinks, 0, sizeof(no_sinks));
        for (int k = ci; k < n; k += 2) {
            const int s = k % kSlots, use = k / kSlots;
            const JacTile T = jac_tile(A, t_begin + k);
            const long long t0 = T.t0;
            const int cnt = T.cnt;
            double *pout = A.out + T.b * A.ostride;
            const bool base_aligned = (reinterpret_cast<uintptr_t>(pout) & 15u) == 0;
            mbar_wait(full_b(s), (unsigned)use & 1u);
            auto release = [&]() { mbar_arrive(empty_b(s)); };
            mma_tile<N_, 4, 0, true, decltype(release)>(slots + (size_t)s * kSlotD, obuf, obuf_s, Bf,
                                                        pout + (size_t)t0 * A.L, no_sinks, t0, cnt, A.L, 0.0, lane,
                                                        base_aligned, false, release);
            __syncwarp();
        }
        if (lane == 0) bulk_wait_all();
    }
}

template <int N_, int DIM, int JMODE> size_t jac_ws_shmem(int L) {
    const size_t slot = (JMODE == J_PAIR_VAR) ? bezws::slot_doubles<N_, DIM>() : bezmma::kRowsDoubles;
    return ((size_t)4 * bezws::kSlots * slot + (size_t)bezws::kConsumers * 16 * L + 4 * bezws::kBarsPerGroup) * sizeof(double);
}

template <int N_, int DIM, int JMODE>
int launch_jac_ws(const bez_plan *plan, const JacArgs &A, cudaStream_t st) {
    FullWeights<N_> FW;
    DiffWeights<N_> DW;
    for (int i = 0; i < (N_ + 1) * (N_ + 1); ++i) FW.w[i] = plan->h_W[i];
    for (int i = 0; i <= N_; ++i) { DW.lo[i] = plan->h_E1lo[i]; DW.hi[i] = plan->h_E1hi[i]; }
    const size_t shmem = jac_ws_shmem<N_, DIM, JMODE>(A.L);
    auto kern = jac_sq_elev_ws_kernel<N_, DIM, JMODE>;
    int sms = 148, per_sm = 1;
    if (int rc = bez_kernel_config((const void *)kern, bezws::kWsThreads, shmem, &sms, &per_sm)) return rc;
    const long long nwt = A.B * A.tpp;
    long long grid = sms;
    if (grid > (nwt + 7) / 8) grid = (nwt + 7) / 8;
    if (grid < 1) return BEZ_OK;
    kern<<<(unsigned)grid, bezws::kWsThreads, shmem, st>>>(A, FW, DW);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

template <int N_, int DIM, int JMODE>
int launch_jac_mma(const bez_plan *plan, const JacArgs &A, cudaStream_t st) {
    FullWeights<N_> FW;
    DiffWeights<N_> DW;
    for (int i = 0; i < (N_ + 1) * (N_ + 1); ++i) FW.w[i] = plan->h_W[i];
    for (int i = 0; i <= N_; ++i) { DW.lo[i] = plan->h_E1lo[i]; DW.hi[i] = plan->h_E1hi[i]; }
    const size_t ws_shmem = jac_ws_shmem<N_, DIM, JMODE>(A.L);
    // Per-variable separation sweep (the 27 GB block of the C4 Jacobian): warp-specialised with a TMA fetch of the
    // partner rows (tools/prof_jac.py: 4.72-4.76 ms in bursts of four launches, 4.39 ms = 0.96 of the HBM peak for an
    // isolated launch under ncu; the 8-warp kernel 4.90 ms).  Without the row fetch (the other modes) one producer
    // cannot feed two consumers -- its stage 1 waits for scattered global loads tile after tile (7.1 ms) -- so they
    // stay on the 8-warp kernel.  BEZGPU_MMA_FLAGS bit 128 keeps everything there (A/B).
    if (JMODE == J_PAIR_VAR && ws_shmem <= 232448 && !(bez_sq_elev_mma_flags() & kFlagNoWarpSpecialisation))
        return launch_jac_ws<N_, DIM, JMODE>(plan, A, st);
    const size_t shmem = (size_t)kWarps * (bezmma::kRowsDoubles + 16 * (size_t)A.L) * sizeof(double);
    auto kern = jac_sq_elev_mma_kernel<N_, DIM, JMODE>;
    int sms = 148, per_sm = 1;
    if (int rc = bez_kernel_config((const void *)kern, kThreads, shmem, &sms, &per_sm)) return rc;
    const long long nwt = A.B * A.tpp;
    long long grid = (long long)sms * per_sm;
    const long long need = (nwt + kWarps - 1) / kWarps;
    if (grid > need) grid = need;
    if (grid < 1) return BEZ_OK;
    kern<<<(unsigned)grid, kThreads, shmem, st>>>(A, FW, DW);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

template <int N_, int DIM, int JMODE>
int launch_jac(const bez_plan *plan, const JacArgs &A, cudaStream_t st) {
    FullWeights<N_> FW;
    DiffWeights<N_> DW;
    for (int i = 0; i < (N_ + 1) * (N_ + 1); ++i) FW.w[i] = plan->h_W[i];
    for (int i = 0; i <= N_; ++i) { DW.lo[i] = plan->h_E1lo[i]; DW.hi[i] = plan->h_E1hi[i]; }
    const size_t shmem = ((size_t)kWarps * 32 * RowGeom<N_>::RS * 2 + (size_t)(2 * N_ + 1) * A.LhPad) * sizeof(double) +
                         (size_t)kWarps * 32 * sizeof(long long);
    if (shmem > 227 * 1024) {
        bez_set_error("degree %d with elevation %d needs %zu bytes of shared memory (> 227 KB)",
                      plan->n, plan->elev, shmem);
        return BEZ_EUNSUPPORTED;
    }
    auto kern = jac_sq_elev_kernel<N_, DIM, JMODE>;
    int sms = 148, per_sm = 1;
    if (int rc = bez_kernel_config((const void *)kern, kThreads, shmem, &sms, &per_sm)) return rc;
    const long long nwt = A.B * A.tpp;
    long long grid = (long long)sms * per_sm;
    const long long need = (nwt + kWarps - 1) / kWarps;
    if (grid > need) grid = need;
    if (grid < 1) return BEZ_OK;
    kern<<<(unsigned)grid, kThreads, shmem, st>>>(A, FW, DW);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

template <int N_, int JMODE>
int jdispatch_dim(const bez_plan *plan, const JacArgs &A, cudaStream_t st) {
    if constexpr (JMODE == J_PAIR_VAR || JMODE == J_SPEED_VAR) {
        const char *e = getenv("BEZGPU_FORCE_DFMA");
        if (!A.dense && A.Lh > 32 && A.Lh <= 64 && !(e && e[0] == '1')) {
            switch (plan->dim) {
                case 1: return launch_jac_mma<N_, 1, JMODE>(plan, A, st);
                case 2: return launch_jac_mma<N_, 2, JMODE>(plan, A, st);
                case 3: return launch_jac_mma<N_, 3, JMODE>(plan, A, st);
            }
        }
    }
    switch (plan->dim) {
        case 1: return launch_jac<N_, 1, JMODE>(plan, A, st);
        case 2: return launch_jac<N_, 2, JMODE>(plan, A, st);
        case 3: return launch_jac<N_, 3, JMODE>(plan, A, st);
    }
    return BEZ_EUNSUPPORTED;
}

template <int JMODE>
int jdispatch(const bez_plan *plan, const JacArgs &A, cudaStream_t st) {
    switch (plan->n) {
#define CASE(n_) case n_: return jdispatch_dim<n_, JMODE>(plan, A, st);
#ifdef BEZ_ONLY_N   /* development builds: one degree only (fast compile) */
        CASE(BEZ_ONLY_N)
#else
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
        CASE(9) CASE(10) CASE(11) CASE(12)
#endif
#undef CASE
    }
    bez_set_error("degree %d has no Jacobian kernel instantiation (1..12 supported)", plan->n);
    return BEZ_EUNSUPPORTED;
}

}  // namespace

// literal 2-point quotient for constraints without a closed form (angular rate), per sweep p:
//   JT[p][k][r] = (F[p][k+1][r] - F[p][0][r]) / dx[p][k]      (_numdiff.py:709-711)
static __global__ void fd_quotient_batched_kernel(const double *__restrict__ F, const double *__restrict__ dx,
                                           long long count, int nvar, long long m, double *__restrict__ JT) {
    const long long per = (long long)nvar * m, total = count * per;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / per, rem = idx - p * per;
        const long long k = rem / m, r = rem - k * m;
        const double *Fp = F + p * (nvar + 1) * m;
        JT[idx] = __ddiv_rn(__dsub_rn(Fp[(k + 1) * m + r], Fp[r]), __ldg(dx + p * nvar + k));
    }
}

extern "C" int bez_fd_quotient_batched(const double *d_F, const double *d_dx, int64_t count, int nvar,
                                       int64_t m, double *d_JT, void *stream) {
    BEZ_REQUIRE(d_F && d_dx && d_JT, "NULL argument");
    BEZ_REQUIRE(count >= 0 && nvar >= 0 && m >= 0, "negative size");
    if (count == 0 || nvar == 0 || m == 0) return BEZ_OK;
    long long blocks = ((long long)count * nvar * m + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    fd_quotient_batched_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(d_F, d_dx, count, nvar, m, d_JT);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

extern "C" int bez_fd_quotient(const double *d_F, const double *d_dx, int nvar, int64_t m,
                               double *d_JT, void *stream) {
    return bez_fd_quotient_batched(d_F, d_dx, 1, nvar, m, d_JT, stream);
}

namespace {

// Zero `len` doubles at out + b * stride + off for every point b (rows no item writes).
__global__ void zero_rows_kernel(double *__restrict__ out, long long B, long long stride, long long off,
                                 long long len) {
    const long long total = B * len;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / len;
        out[b * stride + off + (idx - b * len)] = 0.0;
    }
}

int zero_rows(double *out, long long B, long long stride, long long off, long long len, cudaStream_t st) {
    if (B == 0 || len == 0) return BEZ_OK;
    if (stride == len && off == 0) {
        BEZ_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)(B * len), st));
        return BEZ_OK;
    }
    long long blocks = (B * len + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    zero_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(out, B, stride, off, len);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

// Shared body of the separation entries.  With one vehicle, the leading N-1 pairs and ld = (N-1)*L,
// item (kk, uu) of the dense J^T lands at kk*ld + uu*L and the tf rows at kdir*ld: a point's dense
// block is its sweep block byte for byte, nothing is left to zero, and the dense request runs as a
// sweep (on the tensor path where L allows).  kdir >= 0 with d_dir == NULL: tf moves no control
// point, its rows are 0.
int jac_sep_impl(const bez_plan *plan, const double *d_cpts, long long B, int N, int numVeh, int ncols,
                 int offset, const double *d_dx, const double *d_dir, int kdir, long long npairs, int dense,
                 double *d_out, int64_t ld, cudaStream_t st) {
    const long long L = plan->L;
    const long long nvarN = (long long)numVeh * plan->dim * ncols;
    const long long nvar = nvarN + (kdir >= 0 ? 1 : 0);
    const long long S = (plan->dim * (plan->n + 1) + 1) / 2 * 2;
    const long long ndir = kdir >= 0 ? npairs : 0;
    JacArgs A;
    A.early_store = (bez_sq_elev_mma_flags() & kFlagEarlyFence) ? 1 : 0;
    A.cpts = d_cpts; A.dir = d_dir; A.dx = d_dx; A.tfs = nullptr; A.PQ = plan->d_PQ; A.out = d_out;
    A.B = B; A.cstride = (long long)N * S; A.dxstride = nvar; A.ld = ld;
    A.N = N; A.numVeh = numVeh; A.L = plan->L; A.Lh = plan->Lh; A.LhPad = plan->LhPad;
    A.ncols = ncols; A.offset = offset; A.kdir = kdir; A.tf = 1.0; A.scale = 0.5 * plan->dim;
    A.dense = dense && !(numVeh == 1 && npairs == N - 1 && ld == npairs * L);
    A.ostride = A.dense ? nvar * ld : (nvarN * (N - 1) + ndir) * L;
    if (A.dense && (numVeh > 1 || npairs > N - 1 || ld > npairs * L)) {
        // rows of pairs without the variable's vehicle are never written
        BEZ_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * (size_t)(B * nvar * ld), st));
    } else if (kdir >= 0 && !d_dir) {
        // the tf rows: J^T row kdir (dense) or the trailing npairs rows (sweep)
        const long long off = A.dense ? (long long)kdir * ld : nvarN * (N - 1) * L;
        if (int rc = zero_rows(d_out, B, A.ostride, off, A.dense ? ld : ndir * L, st)) return rc;
    }
    A.nitems = nvarN * (N - 1);
    A.tpp = (A.nitems + 31) / 32;
    if (A.nitems > 0) {
        int rc = jdispatch<J_PAIR_VAR>(plan, A, st);
        if (rc != BEZ_OK) return rc;
    }
    if (kdir >= 0 && d_dir && npairs > 0) {
        if (!A.dense) A.out = d_out + (size_t)A.nitems * L;
        A.nitems = npairs;
        A.tpp = (A.nitems + 31) / 32;
        return jdispatch<J_PAIR_DIR>(plan, A, st);
    }
    return BEZ_OK;
}

// Shared body of the speed entries; d_tf [B] or NULL (the scalar tf).  One vehicle with ld = L:
// J^T row kk is the sweep row of item kk, the tf row that of vehicle 0, so the dense request runs
// as a sweep.  kdir >= 0 with d_dir == NULL: tf moves no control point, only the n/tf factor.
int jac_speed_impl(const bez_plan *plan, const double *d_cpts, const double *d_tf, double tf, long long B,
                   int N, int numVeh, int ncols, int offset, double alpha, const double *d_dx, const double *d_dir,
                   int kdir, int dense, double *d_out, int64_t ld, cudaStream_t st) {
    const long long L = plan->L;
    const long long nvarN = (long long)numVeh * plan->dim * ncols;
    const long long nvar = nvarN + (kdir >= 0 ? 1 : 0);
    const long long S = (plan->dim * (plan->n + 1) + 1) / 2 * 2;
    JacArgs A;
    A.early_store = (bez_sq_elev_mma_flags() & kFlagEarlyFence) ? 1 : 0;
    A.cpts = d_cpts; A.dir = d_dir; A.dx = d_dx; A.tfs = d_tf; A.PQ = plan->d_PQ; A.out = d_out;
    A.B = B; A.cstride = (long long)N * S; A.dxstride = nvar; A.ld = ld;
    A.N = N; A.numVeh = numVeh; A.L = plan->L; A.Lh = plan->Lh; A.LhPad = plan->LhPad;
    A.ncols = ncols; A.offset = offset; A.kdir = kdir; A.tf = tf; A.scale = alpha * 0.5 * plan->dim;
    A.dense = dense && !(numVeh == 1 && ld == L);
    A.ostride = A.dense ? nvar * ld : (nvarN + (kdir >= 0 ? numVeh : 0)) * L;
    if (A.dense && (numVeh > 1 || ld > (long long)numVeh * L))
        BEZ_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * (size_t)(B * nvar * ld), st));
    A.nitems = nvarN;
    A.tpp = (A.nitems + 31) / 32;
    if (A.nitems > 0) {
        int rc = jdispatch<J_SPEED_VAR>(plan, A, st);
        if (rc != BEZ_OK) return rc;
    }
    if (kdir >= 0) {
        if (!A.dense) A.out = d_out + (size_t)A.nitems * L;
        A.nitems = numVeh;
        A.tpp = (A.nitems + 31) / 32;
        return jdispatch<J_SPEED_DIR>(plan, A, st);
    }
    return BEZ_OK;
}

// Argument checks of the four entries, all before any CUDA call.  ptrs: every pointer the entry
// needs is set; sep: the separation block (its leading npairs pairs), else the speed block.
int jac_check(const bez_plan *plan, bool ptrs, bool sep, long long B, int N, int numVeh, int ncols, int offset,
              int kdir, long long npairs, int dense, int64_t ld) {
    BEZ_REQUIRE(plan && ptrs, "NULL argument");
    BEZ_REQUIRE(B >= 0 && N >= (sep ? 2 : 1) && numVeh >= 1 && numVeh <= N && ncols >= 0 && offset >= 0,
                "bad sizes");
    BEZ_REQUIRE(kdir < 0 || kdir == (long long)numVeh * plan->dim * ncols,
                "kdir must be -1 or the index after the control-point variables");
    const long long P = (long long)N * (N - 1) / 2, nObs = N - numVeh;
    BEZ_REQUIRE(!sep || (npairs >= P - nObs * (nObs - 1) / 2 && npairs <= P),
                "npairs must cover every pair that contains a vehicle and at most all pairs");
    BEZ_REQUIRE(!dense || ld >= (sep ? npairs : numVeh) * (long long)plan->L, "ld smaller than the constraint block");
    if (plan->n < 1 || plan->n > BEZ_MAX_DEGREE_JAC || plan->dim < 1 || plan->dim > 3) {
        bez_set_error("degree %d, dimension %d: the Jacobian kernels cover n <= %d, dim <= 3", plan->n, plan->dim,
                      BEZ_MAX_DEGREE_JAC);
        return BEZ_EUNSUPPORTED;
    }
    return BEZ_OK;
}

}  // namespace

extern "C" int bez_jac_sepsq_elev(const bez_plan *plan, const double *d_cpts, int N, int numVeh,
                                  int ncols, int offset, const double *d_dx, const double *d_dir,
                                  int kdir, int dense, double *d_out, int64_t ld, void *stream) {
    return bez_jac_sepsq_elev_batched(plan, d_cpts, 1, N, numVeh, ncols, offset, d_dx, d_dir, kdir,
                                      (int64_t)N * (N - 1) / 2, dense, d_out, ld, stream);
}

extern "C" int bez_jac_speed_sq_elev(const bez_plan *plan, const double *d_cpts, int N, int numVeh,
                                     int ncols, int offset, double tf, double alpha,
                                     const double *d_dx, const double *d_dir, int kdir, int dense,
                                     double *d_out, int64_t ld, void *stream) {
    if (int rc = jac_check(plan, d_cpts && d_dx && d_out, false, 1, N, numVeh, ncols, offset, kdir, 0, dense, ld))
        return rc;
    BEZ_ON_DEVICE(plan->device);
    return jac_speed_impl(plan, d_cpts, nullptr, tf, 1, N, numVeh, ncols, offset, alpha, d_dx, d_dir, kdir, dense,
                          d_out, ld, (cudaStream_t)stream);
}

extern "C" int bez_jac_sepsq_elev_batched(const bez_plan *plan, const double *d_cpts, int B, int N,
                                          int numVeh, int ncols, int offset, const double *d_dx,
                                          const double *d_dir, int kdir, int64_t npairs, int dense,
                                          double *d_out, int64_t ld, void *stream) {
    if (int rc = jac_check(plan, d_cpts && d_dx && d_out, true, B, N, numVeh, ncols, offset, kdir, npairs, dense, ld))
        return rc;
    if (B == 0) return BEZ_OK;
    BEZ_ON_DEVICE(plan->device);
    return jac_sep_impl(plan, d_cpts, B, N, numVeh, ncols, offset, d_dx, d_dir, kdir, npairs, dense, d_out, ld,
                        (cudaStream_t)stream);
}

extern "C" int bez_jac_speed_sq_elev_batched(const bez_plan *plan, const double *d_cpts, const double *d_tf,
                                             int B, int N, int numVeh, int ncols, int offset, double alpha,
                                             const double *d_dx, const double *d_dir, int kdir, int dense,
                                             double *d_out, int64_t ld, void *stream) {
    if (int rc = jac_check(plan, d_cpts && d_tf && d_dx && d_out, false, B, N, numVeh, ncols, offset, kdir, 0, dense,
                           ld))
        return rc;
    if (B == 0) return BEZ_OK;
    BEZ_ON_DEVICE(plan->device);
    return jac_speed_impl(plan, d_cpts, d_tf, 1.0, B, N, numVeh, ncols, offset, alpha, d_dx, d_dir, kdir, dense,
                          d_out, ld, (cudaStream_t)stream);
}
