// Angular-rate constraint (A6 of SURVEY.md section 8) for sm_100a.
//
// Reference: _maxAngularRateConstraints / _angularRateSqr (optimization.py:425-459,
// 578-611): per 2-D vehicle  pos.elev(E) -> x', x'', y', y'' (Bezier.diff keeps the
// degree m = n+E) -> num = y''*x' - x''*y', den = x'*x' + y'*y' (degree 2m)
// -> num*num / den*den control point by control point (degree 4m).
//
// One CTA per (evaluation point, vehicle); all curves live in shared memory.
// Bernstein products are evaluated as plain convolutions of binomially
// pre-scaled coefficients,  (a*b)_k = sum_i [C(m,i)a_i][C(m,k-i)b_{k-i}] / C(2m,k),
// with the same scipy.special.binom values the reference's weight tables are
// built from (SURVEY Q14).  The degree-2m results are kept pre-scaled for the
// squares, and the common 1/C(4m,k) of numerator and denominator cancels in the
// ratio, so neither the 172 MB dense coefficient matrix of the reference
// (bezier.py:1183-1208 at m = 110) nor C(4m,.) is ever formed.  The squares
// (2 x (2m+1)^2 MACs) use a 4-output register tile with a sliding window so
// that shared-memory traffic is one load per two DFMAs.
//
// Range: coefficient k of a pre-scaled square carries C(4m,k), which runs from 1 at
// the ends to C(4m,2m) ~ 2^(4m) in the middle -- 2^503 at m = 127, 2^995 at m = 250.
// angrate_kernel therefore multiplies its degree-2m rows by 2^-s with
// s = floor(log2 C(4m,2m) / 4) (angrate_v1_shrink), which centres the squares'
// binomial factors on 1: they span 2^-2s .. 2^(log2 C(4m,2m) - 2s), about 2^+-497 at
// m = 250.  The factor is exact and cancels in NUM^2 / DEN^2 (the output does not
// change unless it would leave the fp64 range), and the data's squared numerator and
// denominator may range over about 2^+-525 (1e+-158) at m = 250; unscaled, the middle
// coefficients would overflow once they exceed about 7e8.  The m <= 127 kernels keep
// the unscaled rows: with at most 2^503 in the middle the data keeps 2^520 of headroom.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "angrate_mma.cuh"

namespace {

constexpr int kAThreads = 128;
constexpr int kPad = 4;     // zero padding on both sides of the degree-2m rows

struct AngArgs {
    const double *cpts, *tf;
    const double *Tpos, *lo, *hi, *Cm, *C2m;
    double *out;
    int B, N, S, n, m, veh_begin, nveh;
    double alpha, beta;
};

// shrink = 2^-s of angrate_v1_shrink: applied to the degree-2m rows (see the top of the file)
__global__ void __launch_bounds__(kAThreads) angrate_kernel(const AngArgs A, const double shrink) {
    extern __shared__ __align__(16) double sm[];
    const int m = A.m, n = A.n, m1 = m + 1, L2 = 2 * m + 1;
    double *px = sm, *py = px + m1;
    double *xD = py + m1, *yD = xD + m1, *xDD = yD + m1, *yDD = xDD + m1;
    double *tmpx = yDD + m1, *tmpy = tmpx + m1;
    double *NUM = tmpy + m1 + kPad;                 // [-kPad, L2 + kPad)
    double *DEN = NUM + L2 + 2 * kPad;
    const int tid = threadIdx.x;
    const int b = blockIdx.x / A.nveh;
    const int v = A.veh_begin + (blockIdx.x - b * A.nveh);
    const double *row = A.cpts + ((size_t)b * A.N + v) * A.S;
    const double val = (double)m / __ldg(A.tf + b);            // diffMatrix(m, tf): m/tf

    // pos.elev(E)   (bezier.py:469-495)
    for (int i = tid; i < m1; i += kAThreads) {
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j <= n; ++j) {
            const double t = __ldg(A.Tpos + (size_t)j * m1 + i);
            sx = fma(__ldg(row + j), t, sx);
            sy = fma(__ldg(row + n + 1 + j), t, sy);
        }
        px[i] = sx;
        py[i] = sy;
    }
    for (int i = tid; i < 2 * kPad; i += kAThreads) {
        const int off = (i < kPad) ? (i - kPad) : (L2 + i - kPad);
        NUM[off] = 0.0;
        DEN[off] = 0.0;
    }
    __syncthreads();
    // first derivatives: np.dot(cpts, Dm) then .elev(1)   (bezier.py:497-519)
    for (int k = tid; k < m; k += kAThreads) {
        tmpx[k] = px[k] * (-val) + px[k + 1] * val;
        tmpy[k] = py[k] * (-val) + py[k + 1] * val;
    }
    __syncthreads();
    for (int k = tid; k < m1; k += kAThreads) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        xD[k] = qx;
        yD[k] = qy;
    }
    __syncthreads();
    for (int k = tid; k < m; k += kAThreads) {
        tmpx[k] = xD[k] * (-val) + xD[k + 1] * val;
        tmpy[k] = yD[k] * (-val) + yD[k + 1] * val;
    }
    __syncthreads();
    for (int k = tid; k < m1; k += kAThreads) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k), c = __ldg(A.Cm + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        xDD[k] = qx * c;                      // pre-scale by C(m,k)
        yDD[k] = qy * c;
    }
    __syncthreads();
    for (int k = tid; k < m1; k += kAThreads) {
        const double c = __ldg(A.Cm + k);
        xD[k] *= c;
        yD[k] *= c;
    }
    __syncthreads();
    // degree-2m curves, kept pre-scaled by C(2m,k) and by the exact power of two 2^-s:
    //   NUM = y''*x' - x''*y'      DEN = x'*x' + y'*y'      (optimization.py:603,605)
    for (int k = tid; k < L2; k += kAThreads) {
        const int ilo = k > m ? k - m : 0, ihi = k < m ? k : m;
        double p1 = 0.0, p2 = 0.0, q1 = 0.0, q2 = 0.0;
        for (int i = ilo; i <= ihi; ++i) {
            const double x1 = xD[k - i], y1 = yD[k - i];
            p1 = fma(yDD[i], x1, p1);
            p2 = fma(xDD[i], y1, p2);
            q1 = fma(xD[i], x1, q1);
            q2 = fma(yD[i], y1, q2);
        }
        NUM[k] = (p1 - p2) * shrink;
        DEN[k] = (q1 + q2) * shrink;
    }
    __syncthreads();
    // squares (optimization.py:604,606) and the control-point-wise ratio (:608);
    // 4 consecutive outputs per thread, sliding window over the second factor
    const int L4 = 4 * m + 1;
    double *out = A.out + ((size_t)b * A.nveh + (v - A.veh_begin)) * L4;
    for (int k0 = 4 * tid; k0 < L4; k0 += 4 * kAThreads) {
        const int ilo = k0 > 2 * m ? k0 - 2 * m : 0;
        const int ihi = (k0 + 3) < 2 * m ? (k0 + 3) : 2 * m;
        double nn[4] = {0, 0, 0, 0}, dd[4] = {0, 0, 0, 0};
        double wn[4], wd[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { wn[r] = NUM[k0 + r - ilo]; wd[r] = DEN[k0 + r - ilo]; }
        for (int i = ilo; i <= ihi; ++i) {
            const double an = NUM[i], ad = DEN[i];
#pragma unroll
            for (int r = 0; r < 4; ++r) { nn[r] = fma(an, wn[r], nn[r]); dd[r] = fma(ad, wd[r], dd[r]); }
            wn[3] = wn[2]; wn[2] = wn[1]; wn[1] = wn[0]; wn[0] = NUM[k0 - i - 1];
            wd[3] = wd[2]; wd[2] = wd[1]; wd[1] = wd[0]; wd[0] = DEN[k0 - i - 1];
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (k0 + r < L4) out[k0 + r] = fma(A.alpha, nn[r] / dd[r], A.beta);
    }
}


// ---------------------------------------------------------------------------
// Second-generation kernel: one WARP per (evaluation point, vehicle), register-tiled and
// load-balanced Bernstein products.
//
// A product c_k = sum_i a_i b_{k-i} of two length-La sequences has 2 La - 1 outputs whose term
// counts form a triangle.  Outputs are cut into tiles of R consecutive k; lane j owns tile j
// ("phase A", terms i = 0 .. R j + R - 1) and tile j + H ("phase B", terms i = R (j+H) - La + 1
// .. La - 1): the two term counts add up to the same S = 2 La + R - 1 - R H for every lane, so
// all lanes run the same S steps in lockstep and only the step at which a lane flips from its
// first to its second tile differs (lane j flips at step R (j+1), i.e. exactly one lane flips
// at each R-step segment boundary).  In one step a lane loads one a_i per factor, slides an
// R-wide register window over b (one new element per step) and issues R DFMAs per product:
// R = 8 for the two degree-2m squares (4 LDS : 16 DFMA), R = 4 for the four degree-m products
// (6 LDS : 16 DFMA).  The first kernel spent one LDS per 2 (squares) or 0.7 (products) DFMAs
// and ran at 0.17 of the fp64 pipe on C5.
// Shared-memory rows use the index maps i -> i + i/8 (NUM, DEN) and i -> i + i/4 (derivative
// rows) so that the window loads of 32 lanes, R doubles apart, are bank-conflict free; guard
// zones of zeros around every row stand in for the ragged ends of the triangle.
// Requires ceil((4m+1)/8) <= 64, i.e. m <= 127; larger m uses angrate_kernel.
constexpr int kWarpsW = 4;
constexpr int kGuard = 16;                      // logical guard on both sides of every padded row
                                                // (accessed range, checked for all m <= 127 by emulation:
                                                //  physical offsets [-9, +14] around the row)

__device__ __forceinline__ int pad8(int i) { return i + (i >> 3); }
__device__ __forceinline__ int pad4(int i) { return i + (i >> 2); }

struct WarpPlan {            // host-computed geometry of the two tiled phases
    int H1, nseg1, e1, H2, nseg2, e2;   // e: phase-B start offset in segments (floor, may be -1)
    int lenP4, lenP8;        // doubles per pad4 / pad8 row (with guards)
    int per_warp;            // doubles of shared memory per warp
};

__global__ void __launch_bounds__(32 * kWarpsW, 4) angrate_warp_kernel(const AngArgs A, const WarpPlan W) {
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long item = (long long)blockIdx.x * kWarpsW + warp;
    if (item >= (long long)A.B * A.nveh) return;                 // whole warp; no block-wide barriers below
    const int m = A.m, n = A.n, m1 = m + 1, L2 = 2 * m + 1, L4 = 4 * m + 1;
    double *base = sm + (size_t)warp * W.per_warp;
    double *XD = base + pad4(kGuard);               // logical index i lives at XD[pad4(i)], i >= -kGuard
    double *YD = XD + W.lenP4, *XDD = YD + W.lenP4, *YDD = XDD + W.lenP4;
    double *NUM = YDD + W.lenP4 - pad4(kGuard) + pad8(kGuard);
    double *DEN = NUM + W.lenP8;
    // scratch of the derivative steps lives in the interiors of NUM / DEN (2 m + 1 >= 2 (m + 1) - 1
    // slots each), which phase 1 overwrites completely; the guard zones stay untouched
    double *px = NUM, *py = NUM + m1, *tmpx = DEN, *tmpy = DEN + m1;
    for (int i = lane; i < W.per_warp; i += 32) base[i] = 0.0;   // guard zones (and everything else)
    const int b = (int)(item / A.nveh);
    const int v = A.veh_begin + (int)(item - (long long)b * A.nveh);
    const double *row = A.cpts + ((size_t)b * A.N + v) * A.S;
    const double val = (double)m / __ldg(A.tf + b);              // diffMatrix(m, tf): m/tf
    __syncwarp();

    // pos.elev(E)   (bezier.py:469-495)
    for (int i = lane; i < m1; i += 32) {
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j <= n; ++j) {
            const double t = __ldg(A.Tpos + (size_t)j * m1 + i);
            sx = fma(__ldg(row + j), t, sx);
            sy = fma(__ldg(row + n + 1 + j), t, sy);
        }
        px[i] = sx;
        py[i] = sy;
    }
    __syncwarp();
    // first derivatives: np.dot(cpts, Dm) then .elev(1)   (bezier.py:497-519)
    for (int k = lane; k < m; k += 32) {
        tmpx[k] = px[k] * (-val) + px[k + 1] * val;
        tmpy[k] = py[k] * (-val) + py[k + 1] * val;
    }
    __syncwarp();
    for (int k = lane; k < m1; k += 32) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        px[k] = qx;                                  // x', y' (unscaled) reuse px, py
        py[k] = qy;
    }
    __syncwarp();
    for (int k = lane; k < m; k += 32) {
        tmpx[k] = px[k] * (-val) + px[k + 1] * val;
        tmpy[k] = py[k] * (-val) + py[k + 1] * val;
    }
    __syncwarp();
    for (int k = lane; k < m1; k += 32) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k), c = __ldg(A.Cm + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        XDD[pad4(k)] = qx * c;                       // pre-scaled by C(m,k)
        YDD[pad4(k)] = qy * c;
        XD[pad4(k)] = px[k] * c;
        YD[pad4(k)] = py[k] * c;
    }
    __syncwarp();
    // the scratch rows are dead: clear the NUM / DEN rows (guards included) for phase 1
    for (int i = lane; i < 2 * W.lenP8; i += 32) (NUM - pad8(kGuard))[i] = 0.0;
    __syncwarp();

    // Addressing: with the phase-B start rounded down to a multiple of R (e1, e2 below; the
    // extra leading terms hit window zeros) every index of a segment is "multiple of R plus u",
    // so under the maps i -> i + i/R the loads of a segment are  pointer[+-u]  with one pointer
    // update per row and segment instead of shift/add index arithmetic per load.
    // ---- phase 1: NUM = y''*x' - x''*y', DEN = x'*x' + y'*y' (pre-scaled by C(2m,k)), R = 4
    {
        constexpr int R = 4, P = R + 1;              // P = padded stride of one segment
        const bool active = lane < W.H1;
        const int j = active ? lane : W.H1 - 1;
        int k0 = R * j;
        double num[R], den[R], wx[R], wy[R];
        const double *ax = XD, *ay = YD, *axx = XDD, *ayy = YDD;   // a side: row[P (q + ea) + u]
        const double *bx = XD + P * j - 2, *by = YD + P * j - 2;   // window:  row[P (jw - q) - 2 - u]
#pragma unroll
        for (int r = 0; r < R; ++r) {
            num[r] = 0.0; den[r] = 0.0;
            wx[r] = bx[2 + r];
            wy[r] = by[2 + r];
        }
        for (int q = 0; q < W.nseg1; ++q) {
            if (q == j + 1) {                        // this lane flips to its second tile
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (active && k0 + r < L2) { NUM[pad8(k0 + r)] = num[r]; DEN[pad8(k0 + r)] = den[r]; }
                k0 = R * (j + W.H1);
                ax += P * W.e1; ay += P * W.e1; axx += P * W.e1; ayy += P * W.e1;
                bx += P * (W.H1 - W.e1); by += P * (W.H1 - W.e1);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    num[r] = 0.0; den[r] = 0.0;
                    wx[r] = bx[2 + r];
                    wy[r] = by[2 + r];
                }
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const double ydd = ayy[u], xdd = axx[u], xd = ax[u], yd = ay[u];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const double vx = wx[(r - u) & (R - 1)], vy = wy[(r - u) & (R - 1)];
                    num[r] = fma(ydd, vx, num[r]);
                    num[r] = fma(-xdd, vy, num[r]);
                    den[r] = fma(xd, vx, den[r]);
                    den[r] = fma(yd, vy, den[r]);
                }
                wx[(R - 1 - u) & (R - 1)] = bx[-u];
                wy[(R - 1 - u) & (R - 1)] = by[-u];
            }
            ax += P; ay += P; axx += P; ayy += P;
            bx -= P; by -= P;
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (active && k0 + r < L2) { NUM[pad8(k0 + r)] = num[r]; DEN[pad8(k0 + r)] = den[r]; }
    }
    __syncwarp();

    // ---- phase 2: squares (optimization.py:604,606) and the control-point-wise ratio (:608), R = 8
    {
        constexpr int R = 8, P = R + 1;
        double *out = A.out + (size_t)item * L4;
        const bool active = lane < W.H2;
        const int j = active ? lane : W.H2 - 1;
        int k0 = R * j;
        double nn[R], dd[R], wn[R], wd[R];
        double nnA[R], ddA[R];                       // results of the first tile, divided at the end
        const int k0A = k0;
        const double *an_ = NUM, *ad_ = DEN;
        const double *bn = NUM + P * j - 2, *bd = DEN + P * j - 2;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            nn[r] = 0.0; dd[r] = 0.0; nnA[r] = 0.0; ddA[r] = 1.0;
            wn[r] = bn[2 + r];
            wd[r] = bd[2 + r];
        }
        bool flipped = false;
        for (int q = 0; q < W.nseg2; ++q) {
            if (q == j + 1) {
                // one lane at a time runs this block: keep it short (the divisions wait until
                // every lane can do them together)
#pragma unroll
                for (int r = 0; r < R; ++r) { nnA[r] = nn[r]; ddA[r] = dd[r]; }
                flipped = true;
                k0 = R * (j + W.H2);
                an_ += P * W.e2; ad_ += P * W.e2;
                bn += P * (W.H2 - W.e2); bd += P * (W.H2 - W.e2);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    nn[r] = 0.0; dd[r] = 0.0;
                    wn[r] = bn[2 + r];
                    wd[r] = bd[2 + r];
                }
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const double an = an_[u], ad = ad_[u];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    nn[r] = fma(an, wn[(r - u) & (R - 1)], nn[r]);
                    dd[r] = fma(ad, wd[(r - u) & (R - 1)], dd[r]);
                }
                wn[(R - 1 - u) & (R - 1)] = bn[-u];
                wd[(R - 1 - u) & (R - 1)] = bd[-u];
            }
            an_ += P; ad_ += P;
            bn -= P; bd -= P;
        }
        if (!flipped) {                              // (last lane when the segment count equals H2)
#pragma unroll
            for (int r = 0; r < R; ++r) { nnA[r] = nn[r]; ddA[r] = dd[r]; nn[r] = 0.0; dd[r] = 1.0; }
            k0 = L4;                                 // nothing to write for a second tile
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (active && k0A + r < L4) out[k0A + r] = fma(A.alpha, nnA[r] / ddA[r], A.beta);
            if (active && k0 + r < L4) out[k0 + r] = fma(A.alpha, nn[r] / dd[r], A.beta);
        }
    }
}

// ---------------------------------------------------------------------------
// Third generation: the same balanced tiling, but the two half-warps work on different
// products so that a lane needs fewer shared-memory loads per DFMA (ncu on the kernel above:
// L1 data pipe 85 %, fp64 pipe 49 % -- every LDS.64 of a warp moves 256 bytes to the
// register file whatever its address pattern).
//   phase 1 (R = 8):  lanes 0..15 NUM = y''*x' + (-x'')*y',  lanes 16..31 DEN = x'*x' + y'*y'
//                     4 loads : 16 DFMA per step   (was 6 : 16)
//   phase 2 (R = 16): lanes 0..15 NUM^2,  lanes 16..31 DEN^2
//                     2 loads : 16 DFMA per step   (was 4 : 16)
// Lane j of a half owns tiles j and j + H (H <= 16 for m <= 127); the ratio needs one
// exchange of 16 values with the partner lane (shfl xor 16) at the very end.
constexpr int kGuard2 = 32;
__device__ __forceinline__ int pad16(int i) { return i + (i >> 4); }

struct WarpPlan2 {
    int H1, nseg1, e1, H2, nseg2, e2;
    int lenP8, lenP16;       // doubles per pad8 / pad16 row (with guards)
    int per_warp;
};

__global__ void __launch_bounds__(32 * kWarpsW, 4) angrate_warp2_kernel(const AngArgs A, const WarpPlan2 W) {
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long item = (long long)blockIdx.x * kWarpsW + warp;
    if (item >= (long long)A.B * A.nveh) return;                 // whole warp; no block-wide barriers below
    const int m = A.m, n = A.n, m1 = m + 1, L2 = 2 * m + 1, L4 = 4 * m + 1;
    double *base = sm + (size_t)warp * W.per_warp;
    double *XD = base + pad8(kGuard2);              // logical index i lives at XD[pad8(i)], i >= -kGuard2
    double *YD = XD + W.lenP8, *XDN = YD + W.lenP8, *YDD = XDN + W.lenP8;      // XDN = -x''
    double *NUM = YDD + W.lenP8 - pad8(kGuard2) + pad16(kGuard2);              // pad16 rows
    double *DEN = NUM + W.lenP16;
    double *px = NUM, *py = NUM + m1, *tmpx = DEN, *tmpy = DEN + m1;           // scratch, cleared below
    for (int i = lane; i < W.per_warp; i += 32) base[i] = 0.0;
    const int b = (int)(item / A.nveh);
    const int v = A.veh_begin + (int)(item - (long long)b * A.nveh);
    const double *row = A.cpts + ((size_t)b * A.N + v) * A.S;
    const double val = (double)m / __ldg(A.tf + b);              // diffMatrix(m, tf): m/tf
    __syncwarp();

    // pos.elev(E)   (bezier.py:469-495)
    for (int i = lane; i < m1; i += 32) {
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j <= n; ++j) {
            const double t = __ldg(A.Tpos + (size_t)j * m1 + i);
            sx = fma(__ldg(row + j), t, sx);
            sy = fma(__ldg(row + n + 1 + j), t, sy);
        }
        px[i] = sx;
        py[i] = sy;
    }
    __syncwarp();
    // first derivatives: np.dot(cpts, Dm) then .elev(1)   (bezier.py:497-519)
    for (int k = lane; k < m; k += 32) {
        tmpx[k] = px[k] * (-val) + px[k + 1] * val;
        tmpy[k] = py[k] * (-val) + py[k + 1] * val;
    }
    __syncwarp();
    for (int k = lane; k < m1; k += 32) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        px[k] = qx;                                  // x', y' (unscaled) reuse px, py
        py[k] = qy;
    }
    __syncwarp();
    for (int k = lane; k < m; k += 32) {
        tmpx[k] = px[k] * (-val) + px[k + 1] * val;
        tmpy[k] = py[k] * (-val) + py[k + 1] * val;
    }
    __syncwarp();
    for (int k = lane; k < m1; k += 32) {
        const double lo = __ldg(A.lo + k), hi = __ldg(A.hi + k), c = __ldg(A.Cm + k);
        double qx = (k < m) ? tmpx[k] * lo : 0.0, qy = (k < m) ? tmpy[k] * lo : 0.0;
        if (k > 0) { qx = tmpx[k - 1] * hi + qx; qy = tmpy[k - 1] * hi + qy; }
        XDN[pad8(k)] = -(qx * c);                    // pre-scaled by C(m,k); x'' stored negated
        YDD[pad8(k)] = qy * c;
        XD[pad8(k)] = px[k] * c;
        YD[pad8(k)] = py[k] * c;
    }
    __syncwarp();
    for (int i = lane; i < 2 * W.lenP16; i += 32) (NUM - pad16(kGuard2))[i] = 0.0;   // scratch rows are dead
    __syncwarp();

    const int half = lane >> 4, jl = lane & 15;
    // ---- phase 1 (R = 8): acc_k = sum_i p_i x'_{k-i} + q_i y'_{k-i},  (p, q) = (y'', -x'') or (x', y')
    {
        constexpr int R = 8, P = R + 1;
        const bool active = jl < W.H1;
        const int j = active ? jl : W.H1 - 1;
        int k0 = R * j;
        double acc[R], wx[R], wy[R];
        const double *ap = half ? XD : YDD, *aq = half ? YD : XDN;          // a side: row[P (q + ea) + u]
        const double *bx = XD + P * j - 2, *by = YD + P * j - 2;            // window:  row[P (jw - q) - 2 - u]
        double *dst = half ? DEN : NUM;
#pragma unroll
        for (int r = 0; r < R; ++r) { acc[r] = 0.0; wx[r] = bx[2 + r]; wy[r] = by[2 + r]; }
        for (int q = 0; q < W.nseg1; ++q) {
            if (q == j + 1) {                        // this lane flips to its second tile
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (active && k0 + r < L2) dst[pad16(k0 + r)] = acc[r];
                k0 = R * (j + W.H1);
                ap += P * W.e1; aq += P * W.e1;
                bx += P * (W.H1 - W.e1); by += P * (W.H1 - W.e1);
#pragma unroll
                for (int r = 0; r < R; ++r) { acc[r] = 0.0; wx[r] = bx[2 + r]; wy[r] = by[2 + r]; }
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const double pv = ap[u], qv = aq[u];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    acc[r] = fma(pv, wx[(r - u) & (R - 1)], acc[r]);
                    acc[r] = fma(qv, wy[(r - u) & (R - 1)], acc[r]);
                }
                wx[(R - 1 - u) & (R - 1)] = bx[-u];
                wy[(R - 1 - u) & (R - 1)] = by[-u];
            }
            ap += P; aq += P;
            bx -= P; by -= P;
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (active && k0 + r < L2) dst[pad16(k0 + r)] = acc[r];
    }
    __syncwarp();

    // ---- phase 2 (R = 16): squares (optimization.py:604,606); ratio (:608) after one exchange
    {
        constexpr int R = 16, P = R + 1;
        double *out = A.out + (size_t)item * L4;
        const bool active = jl < W.H2;
        const int j = active ? jl : W.H2 - 1;
        int k0 = R * j;
        const int k0A = k0;
        double acc[R], w[R], accA[R];
        const double *src = half ? DEN : NUM;
        const double *ap = src;
        const double *bw = src + P * j - 2;
#pragma unroll
        for (int r = 0; r < R; ++r) { acc[r] = 0.0; accA[r] = 0.0; w[r] = bw[2 + r]; }
        bool flipped = false;
        for (int q = 0; q < W.nseg2; ++q) {
            if (q == j + 1) {
#pragma unroll
                for (int r = 0; r < R; ++r) accA[r] = acc[r];
                flipped = true;
                k0 = R * (j + W.H2);
                ap += P * W.e2;
                bw += P * (W.H2 - W.e2);
#pragma unroll
                for (int r = 0; r < R; ++r) { acc[r] = 0.0; w[r] = bw[2 + r]; }
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const double av = ap[u];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = fma(av, w[(r - u) & (R - 1)], acc[r]);
                w[(R - 1 - u) & (R - 1)] = bw[-u];
            }
            ap += P;
            bw -= P;
        }
        if (!flipped) {                              // (last lane when the segment count equals H2)
#pragma unroll
            for (int r = 0; r < R; ++r) { accA[r] = acc[r]; acc[r] = 0.0; }
            k0 = L4;                                 // no second tile
        }
        // half 0 holds NUM^2 (tiles A, B), half 1 DEN^2: half 0 finishes tile A, half 1 tile B
        const int kB = __shfl_xor_sync(0xffffffffu, k0, 16);       // (equal in both halves)
        (void)kB;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const double other = __shfl_xor_sync(0xffffffffu, half ? accA[r] : acc[r], 16);
            // half 0: other = DEN^2 of tile A;  half 1: other = NUM^2 of tile B
            const double nn = half ? other : accA[r];
            const double dd = half ? acc[r] : other;
            const int k = (half ? k0 : k0A) + r;
            if (active && k < L4) out[k] = fma(A.alpha, nn / dd, A.beta);
        }
    }
}

// ---------------------------------------------------------------------------
// Fourth generation: the Bernstein products on the fp64 tensor path (DMMA.8x8x4), operands in
// registers, squares at half cost.
//
// ncu on the third generation (profiles/r01_ncu_angrate_warp_kernel.txt): L1 data pipe 85 %,
// fp64 pipe 49 % -- the sliding-window convolution streams its operands through LDS.  A
// convolution c_k = sum_i a_i b_{k-i} has no shared operand between outputs, but cut into blocks
// of 8 it becomes a sum of 8 x 8 outer products: with A_u = (a_{8u+g})_g, B_v = (b_{8v+j})_j,
//     C_w[g][j] = sum_u a_{8u+g} b_{8(w-u)+j}            (an 8 x U times U x 8 GEMM over u)
//     c_{8w+s}  = sum_{g+j=s} C_w[g][j]  (+ the part of C_{w-1} with g + j = s + 8)
// One DMMA covers four u; in fragment form lane (g,t) needs a_{8(4q+t)+g} for the q-th k-step
// (independent of w) and b_{8(w-4q-t)+g} (a function of w - 4q): the whole of a and b lives in
// U/4 + U + 3 registers per lane and NO operand is loaded inside the product loops (all loop
// bounds are compile-time, every register index is static).
// Squares (three of the four product groups: x'x' + y'y', NUM^2, DEN^2): the outer products of
// (u, v) and (v, u) are transposes of each other and have the same anti-diagonal sums, so only
// u < w/2 is computed (plus half of the diagonal block u = w/2); the result is half the true
// value, an exact scaling that cancels in NUM^2 / DEN^2 and is undone for DEN by an exact x 2.
// Anti-diagonal sums: the C fragments of two blocks at a time are scattered into a 32-row ring
// Z[row = k mod 32][slot = g] in shared memory (every slot is written exactly once per output row:
// slots g <= s by block w, g > s by block w - 1), then 16 lanes sum the 16 finished rows (ring_pair).
// Per vehicle 482 DMMA + 84 ring passes instead of 4600 warp-wide DFMA + 9000 LDS.
// Instantiated per block count U1 = ceil((m+1)/8) (U2 = 2 U1 blocks for the degree-2m curves).
constexpr int kMmaWarps = 4;
template <int U1>
__global__ void __launch_bounds__(32 * kMmaWarps, 4) angrate_mma_kernel(const AngArgs A) {
    constexpr int U2 = 2 * U1;
    constexpr int ROW1 = kMmaGuard + 8 * U1 + kMmaGuard + 8;       // operand row of a degree-m curve
    constexpr int ROW2 = kMmaGuard + 8 * U2 + kMmaGuard + 8;       // ... of a degree-2m curve
    constexpr int PER_WARP = 4 * ROW1 + 2 * ROW2 + kRingDoubles;
    static_assert(4 * ROW1 >= 16 * U2 && 2 * ROW2 >= 16 * U2, "result rows alias the dead operand rows");
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const long long item = (long long)blockIdx.x * kMmaWarps + warp;
    if (item >= (long long)A.B * A.nveh) return;                 // whole warp; no block-wide barriers below
    const int m = A.m, n = A.n, m1 = m + 1, L4 = 4 * m + 1;
    double *base = sm + (size_t)warp * PER_WARP;
    double *XD = base + kMmaGuard, *YD = XD + ROW1, *XDN = YD + ROW1, *YDD = XDN + ROW1;   // XDN = -x''
    double *NUM = base + 4 * ROW1 + kMmaGuard, *DEN = NUM + ROW2;
    double *Z = base + 4 * ROW1 + 2 * ROW2;                       // [32][8] ring
    double *N2 = base;                                            // NUM^2 (16 U2 doubles) over the dead degree-m rows
    double *D2 = base + 4 * ROW1;                                 // DEN^2 over the dead NUM | DEN rows
    double *px = NUM, *py = NUM + 8 * U1;                         // scratch (cleared below)
    for (int i = lane; i < PER_WARP; i += 32) base[i] = 0.0;
    const int b = (int)(item / A.nveh);
    const int v = A.veh_begin + (int)(item - (long long)b * A.nveh);
    const double *row = A.cpts + ((size_t)b * A.N + v) * A.S;
    const double val = (double)m / __ldg(A.tf + b);              // diffMatrix(m, tf): m/tf
    __syncwarp();

    // pos.elev(E)   (bezier.py:469-495); the 2 (n+1) control points go through the (still unused) ring
    // so that every lane reads them as shared-memory broadcasts instead of 2 (n+1) global loads per output
    for (int j = lane; j < 2 * (n + 1); j += 32) Z[j] = __ldg(row + j);
    __syncwarp();
    for (int i = lane; i < m1; i += 32) {
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j <= n; ++j) {
            const double tt = __ldg(A.Tpos + (size_t)j * m1 + i);
            sx = fma(Z[j], tt, sx);
            sy = fma(Z[n + 1 + j], tt, sy);
        }
        px[i] = sx;
        py[i] = sy;
    }
    __syncwarp();
    for (int j = lane; j < 2 * (n + 1); j += 32) Z[j] = 0.0;       // the ring starts zeroed
    __syncwarp();
    // first and second derivatives in one pass (diff2_stencil, angrate_mma.cuh)
    for (int k = lane; k < m1; k += 32) {
        const double *rows[2] = {px, py};
        double d1[2], d2[2];
        diff2_stencil<2>(rows, A.lo, A.hi, k, m, val, d1, d2);
        const double c = __ldg(A.Cm + k);
        XDN[k] = -(d2[0] * c);                       // pre-scaled by C(m,k); x'' stored negated
        YDD[k] = d2[1] * c;
        XD[k] = d1[0] * c;
        YD[k] = d1[1] * c;
    }
    __syncwarp();
    for (int i = lane; i < 2 * ROW2; i += 32) (NUM - kMmaGuard)[i] = 0.0;        // scratch is dead: clear the rows
    __syncwarp();

    // ---- degree-2m curves, pre-scaled by C(2m,k) (optimization.py:603,605)
    {
        ConvRegs<U1> R1, R2;
        conv_load<U1>(R1, YDD, XD, g, t);            // y'' * x'
        conv_load<U1>(R2, XDN, YD, g, t);            // (-x'') * y'
        conv_all<U1, false, true, (U1 % 2 == 1)>(R1, R2, Z, NUM, 1.0, g, t, lane);
        conv_load<U1>(R1, XD, XD, g, t);             // x' * x'
        conv_load<U1>(R2, YD, YD, g, t);             // y' * y'
        conv_all<U1, true, true, (U1 % 2 == 1)>(R1, R2, Z, DEN, 2.0, g, t, lane);   // half squares: exact x 2
    }
    __syncwarp();
    // ---- squares (optimization.py:604,606); both come out halved, which cancels in the ratio
    {
        ConvRegs<U2> R;
        conv_load<U2>(R, NUM, NUM, g, t);
        __syncwarp();
        conv_all<U2, true, false, (U1 % 2 == 1)>(R, R, Z, N2, 1.0, g, t, lane);    // overwrites the degree-m rows
        conv_load<U2>(R, DEN, DEN, g, t);
        __syncwarp();                                                        // operands in registers: rows dead
        conv_all<U2, true, false, (U1 % 2 == 1)>(R, R, Z, D2, 1.0, g, t, lane);
    }
    __syncwarp();
    // ---- control-point-wise ratio (optimization.py:608)
    double *out = A.out + (size_t)item * L4;
    // N2 / D2 with a branch-free division: rcp.approx (2^-23) + two Newton steps + one residual
    // correction of the quotient (the operands are far from the overflow / subnormal ranges that
    // the generic DDIV sequence guards against: |D2| ~ C(2m,.)^4 v^4 stays below 1e260 for m <= 127)
    for (int k = lane; k < L4; k += 32) {
        const double nn = N2[k], dd = D2[k];
        double r;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(dd));
        r = fma(fma(-dd, r, 1.0), r, r);
        r = fma(fma(-dd, r, 1.0), r, r);
        double q = nn * r;
        q = fma(fma(-dd, q, nn), r, q);
        out[k] = fma(A.alpha, q, A.beta);
    }
}

template <int U1>
static int launch_angrate_mma(const AngArgs &A, cudaStream_t st) {
    constexpr int U2 = 2 * U1;
    constexpr int ROW1 = kMmaGuard + 8 * U1 + kMmaGuard + 8, ROW2 = kMmaGuard + 8 * U2 + kMmaGuard + 8;
    const size_t shw = sizeof(double) * (size_t)(4 * ROW1 + 2 * ROW2 + kRingDoubles) * kMmaWarps;
    int sms_ = 0, per_sm_ = 0;
    if (int rc = bez_kernel_config((const void *)angrate_mma_kernel<U1>, 32 * kMmaWarps, shw, &sms_, &per_sm_)) return rc;
    const long long items = (long long)A.B * A.nveh;
    angrate_mma_kernel<U1><<<(unsigned)((items + kMmaWarps - 1) / kMmaWarps), 32 * kMmaWarps, shw, st>>>(A);
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}

static WarpPlan2 make_warp_plan2(int m) {
    WarpPlan2 W;
    const int m1 = m + 1, L2 = 2 * m + 1;
    const int T1 = (2 * m1 - 1 + 7) / 8, T2 = (2 * L2 - 1 + 15) / 16;
    W.H1 = (T1 + 1) / 2;
    W.H2 = (T2 + 1) / 2;
    auto floordiv = [](int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); };
    W.e1 = floordiv(8 * W.H1 - m1 - 7, 8);
    W.e2 = floordiv(16 * W.H2 - L2 - 15, 16);
    W.nseg1 = (m1 - 8 * W.e1 + 7) / 8;
    W.nseg2 = (L2 - 16 * W.e2 + 15) / 16;
    if (W.nseg1 < W.H1) W.nseg1 = W.H1;
    if (W.nseg2 < W.H2) W.nseg2 = W.H2;
    auto p8 = [](int i) { return i + (i >> 3); };
    auto p16 = [](int i) { return i + (i >> 4); };
    W.lenP8 = p8(kGuard2) + p8(m1 + kGuard2) + 2;
    W.lenP16 = p16(kGuard2) + p16(L2 + kGuard2) + 2;
    if (W.lenP16 < p16(kGuard2) + 2 * m1 + 2) W.lenP16 = p16(kGuard2) + 2 * m1 + 2;   // scratch aliasing
    W.per_warp = 4 * W.lenP8 + 2 * W.lenP16 + 8;
    W.per_warp = (W.per_warp + 1) / 2 * 2;
    return W;
}

// 2^-s, s = floor(log2 C(4m,2m) / 4): the scale of angrate_kernel's degree-2m rows
static double angrate_v1_shrink(int m) {
    double l = 0.0;
    for (int k = 1; k <= 2 * m; ++k) l += log2((double)(2 * m + k) / k);    // log2 C(4m,2m)
    return ldexp(1.0, -(int)(l / 4));
}

static WarpPlan make_warp_plan(int m) {
    WarpPlan W;
    const int m1 = m + 1, L2 = 2 * m + 1;
    const int T1 = (2 * m1 - 1 + 3) / 4, T2 = (2 * L2 - 1 + 7) / 8;
    W.H1 = (T1 + 1) / 2;
    W.H2 = (T2 + 1) / 2;
    auto floordiv = [](int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); };
    W.e1 = floordiv(4 * W.H1 - m1 - 3, 4);          // phase B starts at i = 4 (j + 1 + e1)
    W.e2 = floordiv(8 * W.H2 - L2 - 7, 8);
    W.nseg1 = (m1 - 4 * W.e1 + 3) / 4;              // last term i = La - 1 is reached in phase B
    W.nseg2 = (L2 - 8 * W.e2 + 7) / 8;
    if (W.nseg1 < W.H1) W.nseg1 = W.H1;             // every lane must finish its first tile (R H steps)
    if (W.nseg2 < W.H2) W.nseg2 = W.H2;
    auto p4 = [](int i) { return i + (i >> 2); };
    auto p8 = [](int i) { return i + (i >> 3); };
    W.lenP4 = p4(kGuard) + p4(m1 + kGuard) + 2;
    W.lenP8 = p8(kGuard) + p8(L2 + kGuard) + 2;
    if (W.lenP8 < p8(kGuard) + 2 * m1 + 2) W.lenP8 = p8(kGuard) + 2 * m1 + 2;   // scratch aliasing
    W.per_warp = 4 * W.lenP4 + 2 * W.lenP8 + 8;
    W.per_warp = (W.per_warp + 1) / 2 * 2;
    return W;
}

}  // namespace

extern "C" int bez_angrate_tables_create(int n, int elev, int device, const double *h_Tpos,
                                         const double *h_elev1m, const double *h_Cm,
                                         const double *h_C2m, bez_angrate_tables **out) {
    BEZ_REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    BEZ_REQUIRE(h_Tpos && h_elev1m && h_Cm && h_C2m, "tables are NULL");
    BEZ_REQUIRE(n >= 1 && elev >= 0, "bad degree / elevation");
    const int m = n + elev;
    // m <= 250: the squares' binomial factors C(4m,k) 2^-2s span about 2^+-497 at m = 250 (see the
    // top of the file), which leaves the data's squared numerator and denominator about 2^+-525;
    // every extra degree takes 2 bits from both ends
    if (m > 250) {
        bez_set_error("bez_angrate_tables_create: n+elev = %d > 250 (the binomial factors C(4m,k) of the "
                      "degree-4m squares would leave the data too little fp64 range)", m);
        return BEZ_EUNSUPPORTED;
    }
    BEZ_ON_DEVICE(device);
    bez_angrate_tables *t = (bez_angrate_tables *)calloc(1, sizeof(bez_angrate_tables));
    if (!t) { bez_set_error("out of host memory"); return BEZ_ENOMEM; }
    t->n = n; t->elev = elev; t->m = m; t->device = device;
    const int m1 = m + 1;
    double *lo = (double *)malloc(sizeof(double) * m1), *hi = (double *)malloc(sizeof(double) * m1);
    // elevMatrix(m-1,1) is [m][m+1]: q_k = E1[k-1][k] d_{k-1} + E1[k][k] d_k
    for (int k = 0; k < m1; ++k) {
        lo[k] = (k < m) ? h_elev1m[(size_t)k * m1 + k] : 0.0;
        hi[k] = (k > 0) ? h_elev1m[(size_t)(k - 1) * m1 + k] : 0.0;
    }
    cudaError_t e = cudaSuccess;
#define UP(dst, src, cnt)                                                                    \
    if (e == cudaSuccess) e = cudaMalloc((void **)&(dst), sizeof(double) * (cnt));           \
    if (e == cudaSuccess) e = cudaMemcpy((dst), (src), sizeof(double) * (cnt), cudaMemcpyHostToDevice);
    UP(t->d_Tpos, h_Tpos, (size_t)(n + 1) * m1)
    UP(t->d_lo, lo, m1)
    UP(t->d_hi, hi, m1)
    UP(t->d_Cm, h_Cm, m1)
    UP(t->d_C2m, h_C2m, 2 * m + 1)
#undef UP
    free(lo);
    free(hi);
    if (e != cudaSuccess) {
        cudaFree(t->d_Tpos); cudaFree(t->d_lo); cudaFree(t->d_hi); cudaFree(t->d_Cm); cudaFree(t->d_C2m);
        free(t);
        return bez_cuda_fail(e, "angular-rate table upload");
    }
    *out = t;
    return BEZ_OK;
}

extern "C" int bez_angrate_tables_destroy(bez_angrate_tables *t) {
    if (!t) return BEZ_OK;
    cudaFree(t->d_Tpos); cudaFree(t->d_lo); cudaFree(t->d_hi); cudaFree(t->d_Cm); cudaFree(t->d_C2m);
    free(t);
    return BEZ_OK;
}

extern "C" int bez_angrate_sq(const bez_angrate_tables *t, const double *d_cpts, const double *d_tf,
                              int B, int N, int row_stride, int veh_begin, int nveh,
                              double alpha, double beta, double *d_out, void *stream) {
    BEZ_REQUIRE(t && d_cpts && d_tf && d_out, "NULL argument");
    BEZ_REQUIRE(B >= 0 && N >= 0 && veh_begin >= 0 && nveh >= 0 && veh_begin + nveh <= N,
                "vehicle range outside [0, N)");
    BEZ_REQUIRE(row_stride >= 2 * (t->n + 1), "control-point rows are not two dimensional");
    if (B == 0 || nveh == 0) return BEZ_OK;
    BEZ_ON_DEVICE(t->device);
    AngArgs A;
    A.cpts = d_cpts; A.tf = d_tf; A.Tpos = t->d_Tpos; A.lo = t->d_lo; A.hi = t->d_hi;
    A.Cm = t->d_Cm; A.C2m = t->d_C2m; A.out = d_out; A.B = B; A.N = N; A.S = row_stride;
    A.n = t->n; A.m = t->m; A.veh_begin = veh_begin; A.nveh = nveh; A.alpha = alpha; A.beta = beta;
    // BEZGPU_ANGRATE_V1=1 forces the first-generation kernel (A/B runs, tools/check_angrate.py)
    const char *force_v1 = getenv("BEZGPU_ANGRATE_V1");
    const char *gen = getenv("BEZGPU_ANGRATE_GEN");                   // "2" / "3": earlier generations (A/B runs)
    if (!(force_v1 && force_v1[0] == '1') && !(gen && (gen[0] == '2' || gen[0] == '3'))) {
        // fourth generation (DMMA): instantiated for the block counts U1 = ceil((m+1)/8) in use
        switch ((t->m + 1 + 7) / 8) {
#define CASE(u_) case u_: return launch_angrate_mma<u_>(A, (cudaStream_t)stream);
            CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
            CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
            default: break;                                          // m > 127: first-generation kernel
        }
    }
    if (t->m <= 127 && !(force_v1 && force_v1[0] == '1') && !(gen && gen[0] == '2')) {
        const WarpPlan2 W = make_warp_plan2(t->m);                   // half-warp split, R = 8 / 16
        const size_t shw = sizeof(double) * (size_t)W.per_warp * kWarpsW;
        int sms_ = 0, per_sm_ = 0;
        if (int rc = bez_kernel_config((const void *)angrate_warp2_kernel, 32 * kWarpsW, shw, &sms_, &per_sm_)) return rc;
        const long long items = (long long)B * nveh;
        angrate_warp2_kernel<<<(unsigned)((items + kWarpsW - 1) / kWarpsW), 32 * kWarpsW, shw,
                               (cudaStream_t)stream>>>(A, W);
        BEZ_CUDA(cudaGetLastError());
        return BEZ_OK;
    }
    if (t->m <= 127 && !(force_v1 && force_v1[0] == '1')) {           // warp-per-item, tiled and balanced
        const WarpPlan W = make_warp_plan(t->m);
        const size_t shw = sizeof(double) * (size_t)W.per_warp * kWarpsW;
        int sms_ = 0, per_sm_ = 0;
        if (int rc = bez_kernel_config((const void *)angrate_warp_kernel, 32 * kWarpsW, shw, &sms_, &per_sm_)) return rc;
        const long long items = (long long)B * nveh;
        angrate_warp_kernel<<<(unsigned)((items + kWarpsW - 1) / kWarpsW), 32 * kWarpsW, shw,
                              (cudaStream_t)stream>>>(A, W);
        BEZ_CUDA(cudaGetLastError());
        return BEZ_OK;
    }
    const size_t shmem = sizeof(double) * ((size_t)8 * (t->m + 1) + 2 * (2 * t->m + 1 + 2 * kPad) + kPad);
    int sms_ = 0, per_sm_ = 0;
    if (int rc = bez_kernel_config((const void *)angrate_kernel, kAThreads, shmem, &sms_, &per_sm_)) return rc;
    angrate_kernel<<<(unsigned)((long long)B * nveh), kAThreads, shmem, (cudaStream_t)stream>>>(
        A, angrate_v1_shrink(t->m));
    BEZ_CUDA(cudaGetLastError());
    return BEZ_OK;
}
