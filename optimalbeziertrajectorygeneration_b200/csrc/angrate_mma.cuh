// Angular-rate building blocks shared by the evaluation kernel (angrate.cu) and the closed-form
// Jacobian (angrate_jac.cu): the device tables, the fused Bezier.diff-twice stencil and the
// Bernstein products on the fp64 tensor path (DMMA.8x8x4).  The product helpers are described at
// angrate_mma_kernel in angrate.cu.
#pragma once
#include "common.cuh"

struct bez_angrate_tables {
    int n, elev, m, device;
    double *d_Tpos;   // elevMatrix(n, E)           [n+1][m+1]
    double *d_lo;     // elevMatrix(m-1,1)[k][k]     [m+1]
    double *d_hi;     // elevMatrix(m-1,1)[k-1][k]   [m+1]
    double *d_Cm;     // C(m, .)                     [m+1]
    double *d_C2m;    // C(2m, .)                    [2m+1]
};

namespace {

// First and second derivatives of ND degree-m rows at control point k: Bezier.diff =
// np.dot(cpts, Dm) then .elev(1) (bezier.py:497-519), twice, with Dm's entries +-val.  Output k
// needs x'_{k-1..k+1}, i.e. the position control points k-2 .. k+2: every lane recomputes that
// 5-point stencil in registers with exactly the operation order of the separate passes (same
// bits), instead of four passes through shared memory with a warp barrier each.
template <int ND>
__device__ __forceinline__ void diff2_stencil(const double *const (&p)[ND], const double *lo_, const double *hi_,
                                              int k, int m, double val, double (&d1)[ND], double (&d2)[ND]) {
    double P[ND][5];
#pragma unroll
    for (int o = 0; o < 5; ++o) {
        const int j = k - 2 + o;
        const bool in = j >= 0 && j <= m;
#pragma unroll
        for (int q = 0; q < ND; ++q) P[q][o] = in ? p[q][j] : 0.0;
    }
    double lo[3], hi[3];
#pragma unroll
    for (int o = 0; o < 3; ++o) {
        const int j = k - 1 + o;
        const bool in = j >= 0 && j <= m;
        lo[o] = in ? __ldg(lo_ + j) : 0.0;
        hi[o] = in ? __ldg(hi_ + j) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < ND; ++q) {
        double T[4], D[3];
#pragma unroll
        for (int o = 0; o < 4; ++o) {            // tmp_j = p_j (-val) + p_{j+1} val,  j = k-2+o, valid for 0 <= j < m
            const int j = k - 2 + o;
            T[o] = (j >= 0 && j < m) ? P[q][o] * (-val) + P[q][o + 1] * val : 0.0;
        }
#pragma unroll
        for (int o = 0; o < 3; ++o) {            // x'_j, j = k-1+o: tmp_j lo_j (j < m) then + tmp_{j-1} hi_j (j > 0)
            const int j = k - 1 + o;
            double qv = (j >= 0 && j < m) ? T[o + 1] * lo[o] : 0.0;
            if (j > 0 && j <= m) qv = T[o] * hi[o] + qv;
            D[o] = qv;
        }
        d1[q] = D[1];
        const double t0 = (k - 1 >= 0 && k - 1 < m) ? D[0] * (-val) + D[1] * val : 0.0;     // tmp2_{k-1}
        const double t1 = (k < m) ? D[1] * (-val) + D[2] * val : 0.0;                         // tmp2_k
        double qv = (k < m) ? t1 * lo[1] : 0.0;
        if (k > 0) qv = t0 * hi[1] + qv;
        d2[q] = qv;
    }
}

constexpr int kMmaGuard = 32;                   // zeros on both sides of every operand row (doubles)
constexpr int kRingPitch = 10;                  // doubles per ring row (8 slots + 2 pad)
constexpr int kRingDoubles = 32 * kRingPitch;

__device__ __forceinline__ void ang_dmma(double &c0, double &c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int U> struct ConvRegs {
    double a[(U + 3) / 4];          // a[q] = v[8 (4q + t) + g]
    double b[U + 3];                // b[d] = v[8 (d - t) + g]   (zero outside the row: guards)
};
template <int U>
__device__ __forceinline__ void conv_load(ConvRegs<U> &R, const double *va, const double *vb, int g, int t) {
#pragma unroll
    for (int q = 0; q < (U + 3) / 4; ++q) R.a[q] = va[8 * (4 * q + t) + g];
#pragma unroll
    for (int d = 0; d < U + 3; ++d) R.b[d] = vb[8 * (d - t) + g];
}
// One k-step (blocks u = 4Q .. 4Q+3) of block W, if it lies in the block range of W:
//   general product: u in [max(0, W-U+1), min(U-1, W)]
//   SYM (HALF of a square): u < W/2 at weight 1, the diagonal block u = W/2 (W even) at weight 1/2
template <int U, int W, bool SYM>
__device__ __forceinline__ void conv_step(double &c0, double &c1, const ConvRegs<U> &R, int Q, int t) {
    constexpr int ulo = W - (U - 1) > 0 ? W - (U - 1) : 0;
    constexpr int uhi = SYM ? W / 2 : (W < U - 1 ? W : U - 1);
    if (W < 2 * U - 1 && ulo <= uhi && uhi <= U - 1 && Q >= ulo / 4 && Q <= uhi / 4) {
        double bq = R.b[W - 4 * Q];
        if (SYM && Q == uhi / 4) {                       // boundary k-step: drop u > W/2, halve u = W/2 (W even)
            constexpr int ub = uhi % 4;
            if (W % 2 == 0) bq = t > ub ? 0.0 : (t == ub ? 0.5 * bq : bq);
            else bq = t > ub ? 0.0 : bq;
        }
        ang_dmma(c0, c1, R.a[Q], bq);
    }
}

// C fragments of the blocks W and W + 1 (two independent accumulator chains, k-steps interleaved: a
// dependent DMMA costs ~26 cycles, an independent one 16)
template <int U, bool SYM, bool TWO, int W>
__device__ __forceinline__ void conv_pair(double (&cA)[2], double (&cB)[2], const ConvRegs<U> &R1,
                                          const ConvRegs<U> &R2, int t) {
    cA[0] = cA[1] = cB[0] = cB[1] = 0.0;
#pragma unroll
    for (int Q = 0; Q < (U + 3) / 4; ++Q) {
        conv_step<U, W, SYM>(cA[0], cA[1], R1, Q, t);
        conv_step<U, W + 1, SYM>(cB[0], cB[1], R1, Q, t);
        if (TWO) {
            conv_step<U, W, SYM>(cA[0], cA[1], R2, Q, t);
            conv_step<U, W + 1, SYM>(cB[0], cB[1], R2, Q, t);
        }
    }
}

// Ring pass of the block pair (W, W + 1), W even: scatter both C fragments into the 32-row ring
// (row = k mod 32, slot = g: every slot of an output row is written exactly once -- slots g <= s by
// the block the row belongs to, g > s by the block before it), then lanes 0..15 sum the 16 finished
// rows 8W .. 8W+15 and return c_{8W + lane}.
// Row pitch 10 doubles: the 16 lanes of a half-warp (rows R0 + g + 2t, slot g) hit 16 distinct 8-byte
// banks (11 g + 4 t mod 16) -- with pitch 8 every STS was a 4-way conflict and the L1 data pipe sat at
// 96 % (profiles/r02_ncu_angrate_mma_first.txt); the row sums use LDS.128 with 16 active lanes (two
// wavefronts each) and no shuffles, because SHFL shares the L1 data pipe that binds this kernel.
template <int W>
__device__ __forceinline__ double ring_pair(double *Z, const double (&cA)[2], const double (&cB)[2], int g, int t,
                                            int lane) {
    const int k0 = 8 * W + g + 2 * t;
    Z[(k0 & 31) * kRingPitch + g] = cA[0];
    Z[((k0 + 1) & 31) * kRingPitch + g] = cA[1];
    Z[((k0 + 8) & 31) * kRingPitch + g] = cB[0];
    Z[((k0 + 9) & 31) * kRingPitch + g] = cB[1];
    __syncwarp();
    double s = 0.0;
    if (lane < 16) {
        const double2 *zr = reinterpret_cast<const double2 *>(Z + (((8 * W) & 31) + lane) * kRingPitch);
        const double2 v0 = zr[0], v1 = zr[1], v2 = zr[2], v3 = zr[3];
        s = ((v0.x + v0.y) + (v1.x + v1.y)) + ((v2.x + v2.y) + (v3.x + v3.y));
    }
    __syncwarp();                                        // rows 8W .. 8W+6 are rewritten by the next pair
    return s;
}

// dst[8W + r] = scale * (conv(a1, b1) + conv(a2, b2))_{8W + r} for all blocks W = 0 .. 2U-1, two blocks
// per step; the DMMAs of the next pair are issued before the ring pass of this one (its STS -> barrier
// -> LDS chain is pure latency).  CLEAR: the ring rows 0..6 must be zero when a product starts ("block
// -1"); the all-zero last block 2U-1 of the previous product leaves them zero iff U is even.
template <int U, bool SYM, bool TWO, bool CLEAR, int W = 0>
__device__ __forceinline__ void conv_all(const ConvRegs<U> &R1, const ConvRegs<U> &R2, double *Z, double *dst,
                                         double scale, int g, int t, int lane, double a0 = 0.0, double a1 = 0.0,
                                         double b0 = 0.0, double b1 = 0.0) {
    if constexpr (W < 2 * U) {
        double cA[2] = {a0, a1}, cB[2] = {b0, b1};
        if constexpr (W == 0) {
            conv_pair<U, SYM, TWO, 0>(cA, cB, R1, R2, t);
            if constexpr (CLEAR) {
                __syncwarp();                                // the previous product's last ring reads
#pragma unroll
                for (int i = 0; i < kRingDoubles / 32; ++i) Z[32 * i + lane] = 0.0;
                __syncwarp();
            }
        }
        double nA[2] = {0.0, 0.0}, nB[2] = {0.0, 0.0};
        if constexpr (W + 2 < 2 * U) conv_pair<U, SYM, TWO, W + 2>(nA, nB, R1, R2, t);
        const double s = ring_pair<W>(Z, cA, cB, g, t, lane);
        if (lane < 16) dst[8 * W + lane] = s * scale;
        conv_all<U, SYM, TWO, CLEAR, W + 2>(R1, R2, Z, dst, scale, g, t, lane, nA[0], nA[1], nB[0], nB[1]);
    }
}


}  // namespace
