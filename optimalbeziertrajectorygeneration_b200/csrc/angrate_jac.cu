// Closed-form finite-difference Jacobian of the angular-rate block (A6/A7, DESIGN section 3.3).
//
// SciPy's 2-point quotient J_k = (f(x + dx_k e_k) - f(x)) / dx_k of the row
//     f = alpha * s^2 * QQ / SS + beta,   s = m / tf,
//     Q = P(Y2, X1) - P(X2, Y1),  S = P(X1, X1) + P(Y1, Y1),  QQ = P(Q, Q),  SS = P(S, S),
// (P = Bernstein product, X1 / X2 = first / second derivative rows WITHOUT the m/tf factors) is
// formed without cancellation: P is bilinear and symmetric, so P(a', a') - P(a, a) = P(a' - a,
// a' + a), and every difference below is divided by dx_k analytically:
//   control point c of vehicle v, dimension x (y: roles of X and Y swapped), delta = row c of
//   elevMatrix(n, E), dX1 = D delta, dX2 = D^2 delta:
//     dQ = P(Y2, dX1) - P(dX2, Y1)      dS = P(dX1, 2 X1 + dx dX1)
//     dQQ = P(dQ, 2 Q + dx dQ)          dSS = P(dS, 2 S + dx dS)      SS' = SS + dx dSS
//     J = alpha s^2 (dQQ - R dSS) / SS',   R = QQ / SS
//   tf (time-optimal models; the control points move along d_dir, X1_r = D elev(dir_x), ...):
//     dQ = P(Y2_r, X1') + P(Y2, X1_r) - P(X2_r, Y1') - P(X2, Y1_r),   X1' = X1 + dx X1_r
//     dS = P(X1_r, X1 + X1') + P(Y1_r, Y1 + Y1')
//     J = alpha m^2 [ (dQQ - R dSS) / (SS' t'^2) - (2t + dx) R / (t^2 t'^2) ],   t' = t + dx
// Products run on the DMMA helpers of angrate_mma.cuh on binomially pre-scaled rows (the common
// C(4m, k) of dQQ, R dSS and SS' cancels).  Two degree-4m arrays are never multiplied together:
// each sits near C(4m, k) ~ 1e151 at m = 127, and a product of two would overflow fp64.
//
// Pass 1: one warp per (point b, vehicle v) writes the base rows X1, Y1, -X2, Y2 (C(m,.)
// pre-scaled, zero guards included), Q, S (C(2m,.)), R and SS to the caller's scratch.
// Pass 2: one warp per (point b, Jacobian row) reads its vehicle's base rows and writes one
// 4m+1 row.  One warp per row rather than per vehicle: SciPy's closure has B = 1, and a
// two-vehicle problem would otherwise keep two warps busy.
#include "common.cuh"
#include "angrate_mma.cuh"

namespace {

constexpr int kJacWarps = 4;

struct JacAngArgs {
    const double *cpts, *tf, *Tpos, *lo, *hi, *Cm, *dx, *dir;
    double *scratch, *out;
    long long ld;
    int B, N, S, n, m, numVeh, ncols, offset, nvar, kdir, dense, nrows;
    double alpha;
};

template <int U1> struct JacGeom {
    static constexpr int U2 = 2 * U1;
    static constexpr int ROW1 = kMmaGuard + 8 * U1 + kMmaGuard + 8;      // operand row, degree m
    static constexpr int ROW2 = kMmaGuard + 8 * U2 + kMmaGuard + 8;      // ... degree 2m
    static constexpr int L4P = 16 * U2;                                   // degree-4m result row
    static constexpr int SCR = 4 * ROW1 + 2 * ROW2 + 2 * L4P;             // scratch per (b, v)
    static constexpr int BASE_WARP = 4 * ROW1 + 2 * ROW2 + kRingDoubles;  // shared memory per warp
    static constexpr int ROW_WARP = 6 * ROW1 + 5 * ROW2 + kRingDoubles;
    static_assert(SCR == 128 * U1 + 432, "bez_jac_angrate_scratch_doubles documents this count");
    static_assert(6 * ROW1 >= 2 * L4P, "the dQQ | dSS rows alias the dead degree-m rows");
};

// ---- pass 1: base rows of (b, v); the computation of angrate_mma_kernel with s = 1
template <int U1>
__global__ void __launch_bounds__(32 * kJacWarps, 4) angrate_jac_base_kernel(const JacAngArgs A) {
    using G = JacGeom<U1>;
    constexpr int U2 = G::U2, ROW1 = G::ROW1, ROW2 = G::ROW2;
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const long long item = (long long)blockIdx.x * kJacWarps + warp;
    if (item >= (long long)A.B * A.numVeh) return;               // whole warp; no block-wide barriers below
    const int m = A.m, n = A.n, m1 = m + 1, L4 = 4 * m + 1;
    double *base = sm + (size_t)warp * G::BASE_WARP;
    double *XD = base + kMmaGuard, *YD = XD + ROW1, *XDN = YD + ROW1, *YDD = XDN + ROW1;   // XDN = -X2
    double *NUM = base + 4 * ROW1 + kMmaGuard, *DEN = NUM + ROW2;                          // Q, S
    double *Z = base + 4 * ROW1 + 2 * ROW2;
    double *N2 = base, *D2 = base + 4 * ROW1;                     // QQ, SS over dead rows
    double *px = NUM, *py = NUM + 8 * U1;
    for (int i = lane; i < G::BASE_WARP; i += 32) base[i] = 0.0;
    const int b = (int)(item / A.numVeh);
    const int v = (int)(item - (long long)b * A.numVeh);
    const double *row = A.cpts + ((size_t)b * A.N + v) * A.S;
    double *scr = A.scratch + (size_t)item * G::SCR;
    __syncwarp();
    for (int i = lane; i < m1; i += 32) {
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j <= n; ++j) {
            const double tt = __ldg(A.Tpos + (size_t)j * m1 + i);
            sx = fma(__ldg(row + j), tt, sx);
            sy = fma(__ldg(row + n + 1 + j), tt, sy);
        }
        px[i] = sx;
        py[i] = sy;
    }
    __syncwarp();
    for (int k = lane; k < m1; k += 32) {
        const double *rows[2] = {px, py};
        double d1[2], d2[2];
        diff2_stencil<2>(rows, A.lo, A.hi, k, m, 1.0, d1, d2);
        const double c = __ldg(A.Cm + k);
        XDN[k] = -(d2[0] * c);
        YDD[k] = d2[1] * c;
        XD[k] = d1[0] * c;
        YD[k] = d1[1] * c;
    }
    __syncwarp();
    for (int i = lane; i < 2 * ROW2; i += 32) (NUM - kMmaGuard)[i] = 0.0;
    __syncwarp();
    {
        ConvRegs<U1> R1, R2;
        conv_load<U1>(R1, YDD, XD, g, t);
        conv_load<U1>(R2, XDN, YD, g, t);
        conv_all<U1, false, true, (U1 % 2 == 1)>(R1, R2, Z, NUM, 1.0, g, t, lane);    // Q
        conv_load<U1>(R1, XD, XD, g, t);
        conv_load<U1>(R2, YD, YD, g, t);
        conv_all<U1, true, true, (U1 % 2 == 1)>(R1, R2, Z, DEN, 2.0, g, t, lane);     // S (half square x 2)
    }
    __syncwarp();
    for (int i = lane; i < 4 * ROW1 + 2 * ROW2; i += 32) scr[i] = base[i];            // rows with their guards
    __syncwarp();
    {
        ConvRegs<U2> R;
        conv_load<U2>(R, NUM, NUM, g, t);
        __syncwarp();
        conv_all<U2, true, false, (U1 % 2 == 1)>(R, R, Z, N2, 2.0, g, t, lane);       // QQ
        conv_load<U2>(R, DEN, DEN, g, t);
        __syncwarp();
        conv_all<U2, true, false, (U1 % 2 == 1)>(R, R, Z, D2, 2.0, g, t, lane);       // SS
    }
    __syncwarp();
    double *gR = scr + 4 * ROW1 + 2 * ROW2, *gSS = gR + G::L4P;
    for (int k = lane; k < G::L4P; k += 32) {
        gR[k] = k < L4 ? N2[k] / D2[k] : 0.0;
        gSS[k] = k < L4 ? D2[k] : 0.0;
    }
}

// ---- pass 2: one Jacobian row.  TF = false: control-point variables (rows 0 .. numVeh*2*ncols-1
// of the sweep layout, in x's order); TF = true: the tf column, one row per vehicle.
// (two CTAs per SM: the shared memory of the larger instantiations allows no more, and the U2
// products need more than 128 registers there)
template <int U1, bool TF>
__global__ void __launch_bounds__(32 * kJacWarps, 2) angrate_jac_row_kernel(const JacAngArgs A) {
    using G = JacGeom<U1>;
    constexpr int U2 = G::U2, ROW1 = G::ROW1, ROW2 = G::ROW2;
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int nvarN = A.numVeh * 2 * A.ncols;
    const int nitems = TF ? A.numVeh : nvarN;
    const long long item = (long long)blockIdx.x * kJacWarps + warp;
    if (item >= (long long)A.B * nitems) return;                 // whole warp; no block-wide barriers below
    const int m = A.m, n = A.n, m1 = m + 1, L4 = 4 * m + 1;
    double *base = sm + (size_t)warp * G::ROW_WARP;
    double *Z = base;
    double *l1 = base + kRingDoubles + kMmaGuard;                 // local degree-m rows l1 + i ROW1, i < 6
    double *l2 = base + kRingDoubles + 6 * ROW1 + kMmaGuard;      // local degree-2m rows l2 + i ROW2, i < 5
    double *dQQ = base + kRingDoubles, *dSS = dQQ + G::L4P;       // over the dead degree-m rows
    for (int i = lane; i < G::ROW_WARP; i += 32) base[i] = 0.0;
    const int b = (int)(item / nitems);
    const int r = (int)(item - (long long)b * nitems);
    int v, d = 0, c = 0, k;
    if (TF) {
        v = r;
        k = A.kdir;
    } else {
        v = r / (2 * A.ncols);
        const int rem = r - v * 2 * A.ncols;
        d = rem / A.ncols;
        c = A.offset + (rem - d * A.ncols);
        k = r;
    }
    const double *scr = A.scratch + ((size_t)b * A.numVeh + v) * G::SCR;
    const double *gX1 = scr + kMmaGuard, *gY1 = gX1 + ROW1, *gX2N = gY1 + ROW1, *gY2 = gX2N + ROW1;
    const double *gQ = scr + 4 * ROW1 + kMmaGuard, *gS = gQ + ROW2;
    const double *gR = scr + 4 * ROW1 + 2 * ROW2, *gSS = gR + G::L4P;
    const double dx = __ldg(A.dx + (size_t)b * A.nvar + k);
    const double tf = __ldg(A.tf + b);
    double *dQ = l2, *dS = l2 + ROW2, *Qs = l2 + 2 * ROW2, *Ss = l2 + 3 * ROW2, *tmp = l2 + 4 * ROW2;
    __syncwarp();

    if (!TF) {
        // delta = row c of elevMatrix(n, E): the elevated rows of a unit step of control point c
        double *dX1 = l1, *dX2 = l1 + ROW1, *T = l1 + 2 * ROW1;
        for (int i = lane; i < m1; i += 32) tmp[i] = __ldg(A.Tpos + (size_t)c * m1 + i);
        __syncwarp();
        const double *own1 = d ? gY1 : gX1;
        for (int kk = lane; kk < m1; kk += 32) {
            const double *rows[1] = {tmp};
            double d1[1], d2[1];
            diff2_stencil<1>(rows, A.lo, A.hi, kk, m, 1.0, d1, d2);
            const double cm = __ldg(A.Cm + kk);
            dX1[kk] = d1[0] * cm;
            dX2[kk] = d ? d2[0] * cm : -(d2[0] * cm);             // -dX2 for x, +dY2 for y
            T[kk] = fma(dx, dX1[kk], 2.0 * own1[kk]);             // 2 X1 + dx dX1
        }
        __syncwarp();
        ConvRegs<U1> R1, R2;
        if (d == 0) {                                             // P(Y2, dX1) + P(-dX2, Y1)
            conv_load<U1>(R1, gY2, dX1, g, t);
            conv_load<U1>(R2, dX2, gY1, g, t);
        } else {                                                  // P(dY2, X1) + P(-X2, dY1)
            conv_load<U1>(R1, dX2, gX1, g, t);
            conv_load<U1>(R2, gX2N, dX1, g, t);
        }
        conv_all<U1, false, true, true>(R1, R2, Z, dQ, 1.0, g, t, lane);
        conv_load<U1>(R1, dX1, T, g, t);
        conv_all<U1, false, false, true>(R1, R1, Z, dS, 1.0, g, t, lane);
    } else {
        // direction rows: X1_r, Y1_r, -X2_r, Y2_r, then X1', Y1' (later 2 X1 + dx X1_r, 2 Y1 + dx Y1_r)
        double *X1r = l1, *Y1r = l1 + ROW1, *X2Nr = l1 + 2 * ROW1, *Y2r = l1 + 3 * ROW1;
        double *X1p = l1 + 4 * ROW1, *Y1p = l1 + 5 * ROW1;
        if (A.dir) {
            const double *drow = A.dir + (size_t)v * A.S;
            for (int i = lane; i < m1; i += 32) {
                double sx = 0.0, sy = 0.0;
                for (int j = 0; j <= n; ++j) {
                    const double tt = __ldg(A.Tpos + (size_t)j * m1 + i);
                    sx = fma(__ldg(drow + j), tt, sx);
                    sy = fma(__ldg(drow + n + 1 + j), tt, sy);
                }
                tmp[i] = sx;
                tmp[m1 + i] = sy;
            }
        }
        __syncwarp();
        for (int kk = lane; kk < m1; kk += 32) {
            const double *rows[2] = {tmp, tmp + m1};
            double d1[2], d2[2];
            diff2_stencil<2>(rows, A.lo, A.hi, kk, m, 1.0, d1, d2);
            const double cm = __ldg(A.Cm + kk);
            X1r[kk] = d1[0] * cm;
            Y1r[kk] = d1[1] * cm;
            X2Nr[kk] = -(d2[0] * cm);
            Y2r[kk] = d2[1] * cm;
            X1p[kk] = fma(dx, X1r[kk], gX1[kk]);
            Y1p[kk] = fma(dx, Y1r[kk], gY1[kk]);
        }
        __syncwarp();
        ConvRegs<U1> R1, R2;
        conv_load<U1>(R1, Y2r, X1p, g, t);                        // P(Y2_r, X1') + P(Y2, X1_r)
        conv_load<U1>(R2, gY2, X1r, g, t);
        conv_all<U1, false, true, true>(R1, R2, Z, dQ, 1.0, g, t, lane);
        conv_load<U1>(R1, X2Nr, Y1p, g, t);                       // - P(X2_r, Y1') - P(X2, Y1_r)
        conv_load<U1>(R2, gX2N, Y1r, g, t);
        __syncwarp();
        for (int kk = lane; kk < 8 * U1; kk += 32) {              // operands are in registers
            X1p[kk] = fma(dx, X1r[kk], 2.0 * gX1[kk]);
            Y1p[kk] = fma(dx, Y1r[kk], 2.0 * gY1[kk]);
        }
        conv_all<U1, false, true, true>(R1, R2, Z, tmp, 1.0, g, t, lane);
        __syncwarp();
        for (int kk = lane; kk < 16 * U1; kk += 32) dQ[kk] += tmp[kk];
        conv_load<U1>(R1, X1r, X1p, g, t);                        // P(X1_r, X1 + X1') + P(Y1_r, Y1 + Y1')
        conv_load<U1>(R2, Y1r, Y1p, g, t);
        conv_all<U1, false, true, true>(R1, R2, Z, dS, 1.0, g, t, lane);
    }
    __syncwarp();
    for (int kk = lane; kk < 16 * U1; kk += 32) {
        Qs[kk] = fma(dx, dQ[kk], 2.0 * gQ[kk]);                   // Q + Q'
        Ss[kk] = fma(dx, dS[kk], 2.0 * gS[kk]);                   // S + S'
    }
    __syncwarp();
    {
        ConvRegs<U2> R;
        conv_load<U2>(R, dQ, Qs, g, t);
        conv_all<U2, false, false, true>(R, R, Z, dQQ, 1.0, g, t, lane);
        conv_load<U2>(R, dS, Ss, g, t);
        conv_all<U2, false, false, true>(R, R, Z, dSS, 1.0, g, t, lane);
    }
    __syncwarp();
    double *out = A.dense ? A.out + ((size_t)b * A.nvar + k) * (size_t)A.ld + (size_t)v * L4
                          : A.out + ((size_t)b * A.nrows + (TF ? nvarN : 0) + r) * (size_t)L4;
    if (!TF) {
        const double s = (double)m / tf;
        const double f = A.alpha * (s * s);
        for (int kk = lane; kk < L4; kk += 32) {
            const double R = gR[kk], SSp = fma(dx, dSS[kk], gSS[kk]);
            out[kk] = f * (fma(-R, dSS[kk], dQQ[kk]) / SSp);
        }
    } else {
        const double tp = tf + dx, md = (double)m;
        const double f = A.alpha * (md * md), tp2 = tp * tp, c2 = (2.0 * tf + dx) / ((tf * tf) * tp2);
        for (int kk = lane; kk < L4; kk += 32) {
            const double R = gR[kk], SSp = fma(dx, dSS[kk], gSS[kk]);
            out[kk] = f * (fma(-R, dSS[kk], dQQ[kk]) / (SSp * tp2) - c2 * R);
        }
    }
}

template <int U1>
static int launch_angrate_jac(const JacAngArgs &A, cudaStream_t st) {
    using G = JacGeom<U1>;
    const size_t sh1 = sizeof(double) * (size_t)G::BASE_WARP * kJacWarps;
    const size_t sh2 = sizeof(double) * (size_t)G::ROW_WARP * kJacWarps;
    int sms_ = 0, per_sm_ = 0;
    if (int rc = bez_kernel_config((const void *)angrate_jac_base_kernel<U1>, 32 * kJacWarps, sh1, &sms_, &per_sm_)) return rc;
    if (int rc = bez_kernel_config((const void *)angrate_jac_row_kernel<U1, false>, 32 * kJacWarps, sh2, &sms_, &per_sm_)) return rc;
    if (int rc = bez_kernel_config((const void *)angrate_jac_row_kernel<U1, true>, 32 * kJacWarps, sh2, &sms_, &per_sm_)) return rc;
    auto grid = [](long long items) { return (unsigned)((items + kJacWarps - 1) / kJacWarps); };
    angrate_jac_base_kernel<U1><<<grid((long long)A.B * A.numVeh), 32 * kJacWarps, sh1, st>>>(A);
    BEZ_CUDA(cudaGetLastError());
    const long long nvarN = (long long)A.numVeh * 2 * A.ncols;
    if (nvarN > 0) {
        angrate_jac_row_kernel<U1, false><<<grid((long long)A.B * nvarN), 32 * kJacWarps, sh2, st>>>(A);
        BEZ_CUDA(cudaGetLastError());
    }
    if (A.kdir >= 0) {
        angrate_jac_row_kernel<U1, true><<<grid((long long)A.B * A.numVeh), 32 * kJacWarps, sh2, st>>>(A);
        BEZ_CUDA(cudaGetLastError());
    }
    return BEZ_OK;
}

}  // namespace

extern "C" size_t bez_jac_angrate_scratch_doubles(int B, int numVeh, int n, int elev) {
    if (B < 0 || numVeh < 0 || n < 1 || elev < 0 || n + elev > 127) return 0;
    const size_t U1 = (size_t)(n + elev + 1 + 7) / 8;
    return (size_t)B * (size_t)numVeh * (128 * U1 + 432);
}

extern "C" int bez_jac_angrate_sq(const bez_angrate_tables *tables, const double *d_cpts, const double *d_tf,
                                  int B, int N, int row_stride, int numVeh, int ncols, int offset, int nvar,
                                  const double *d_dx, const double *d_dir, int kdir, double alpha, int dense,
                                  double *d_scratch, double *d_out, int64_t ld, void *stream) {
    BEZ_REQUIRE(tables && d_cpts && d_tf && d_dx && d_scratch && d_out, "NULL argument");
    BEZ_REQUIRE(B >= 0 && numVeh >= 1 && numVeh <= N, "vehicle count outside [1, N]");
    BEZ_REQUIRE(row_stride >= 2 * (tables->n + 1), "control-point rows are not two dimensional");
    BEZ_REQUIRE(ncols >= 0 && offset >= 0 && offset + ncols <= tables->n + 1, "free columns outside the curve");
    BEZ_REQUIRE(kdir < 0 || kdir == nvar - 1, "kdir must be the last variable (tf) or -1");
    BEZ_REQUIRE((long long)nvar == (long long)numVeh * 2 * ncols + (kdir >= 0 ? 1 : 0),
                "nvar does not match numVeh * 2 * ncols (+ 1 for tf)");
    const int m = tables->m, L4 = 4 * m + 1;
    BEZ_REQUIRE(!dense || ld >= (long long)numVeh * L4, "ld smaller than the constraint block");
    if (m > 127) {
        bez_set_error("bez_jac_angrate_sq: n+elev = %d > 127 is outside the tensor-path kernels; "
                      "use the literal finite-difference path (bez_fd_quotient)", m);
        return BEZ_EUNSUPPORTED;
    }
    if (B == 0) return BEZ_OK;
    BEZ_ON_DEVICE(tables->device);
    cudaStream_t st = (cudaStream_t)stream;
    JacAngArgs A;
    A.cpts = d_cpts; A.tf = d_tf; A.Tpos = tables->d_Tpos; A.lo = tables->d_lo; A.hi = tables->d_hi;
    A.Cm = tables->d_Cm; A.dx = d_dx; A.dir = kdir >= 0 ? d_dir : nullptr;
    A.scratch = d_scratch; A.out = d_out; A.ld = ld;
    A.B = B; A.N = N; A.S = row_stride; A.n = tables->n; A.m = m; A.numVeh = numVeh; A.ncols = ncols;
    A.offset = offset; A.nvar = nvar; A.kdir = kdir; A.dense = dense;
    A.nrows = numVeh * 2 * ncols + (kdir >= 0 ? numVeh : 0);
    A.alpha = alpha;
    if (dense) BEZ_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * (size_t)B * (size_t)nvar * (size_t)ld, st));
    switch ((m + 1 + 7) / 8) {
#define CASE(u_) case u_: return launch_angrate_jac<u_>(A, st);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
        CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
        default: break;
    }
    return BEZ_EUNSUPPORTED;
}
