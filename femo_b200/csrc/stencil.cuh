// stencil.cuh -- diagonal (DIA) storage of lattice operators for the multigrid V-cycle.
//
// On a lattice mesh every row of the scalar P1 Jacobian couples a node with the same <= 9 relative
// neighbours, so the level matrix is stored as D planes (one per column offset col - row) of fp32 values:
// no column indices, no row pointers, 4*D bytes per row instead of the 8*D + 4 of the fp32 CSR copy, and
// every load of the operator kernel is coalesced with no staging in shared memory.  The planes are a
// re-layout of the assembled (BC'd) CSR values, so the operator is the same matrix the reference would
// factorise (femo/fea/utils_dolfinx.py:476-512) rounded to fp32 -- used inside the preconditioner only.
//
// Row epilogues: the Chebyshev smoother steps of multigrid.cuh are fused into the operator, the
// Jacobi scaling 1/a_ii is taken from the diagonal plane (no dinv vector), the zero-guess degree-2
// pre-smoother is ONE kernel, and residual/direction vectors that nobody reads are not written.
// k_dia_apply serves the V-cycle of multi-GPU slab levels, levels without a 2:1 nested coarse level, the other smoother
// degrees and the residuals of the full-multigrid start; single-GPU levels above the cooperative coarse kernel's range
// run the same row arithmetic inside the two level sweeps of mgsweep.cuh.
//
// Included by engine.cu after SpmvEpi is defined.
#pragma once
#include "common.cuh"

namespace femo {

// CSR (fp64) -> DIA planes (fp32); entries absent from the CSR row are stored as 0.  `bad` is raised when an
// entry's offset is not in the table (the host checked the pattern, so this never fires on a sane layout).
// The same pass yields what the smoother set-up needs from the fp64 values: dinv_i = 1/a_ii and the per-CTA maximum of
// the Gershgorin bound sum_j |a_ij| / |a_ii| over the owned rows [o0,o1) (partials[blockIdx.x]).
template <int D>
__global__ void __launch_bounds__(kThreads)
    k_csr_to_dia(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ vals,
                 DiaMat A, float *__restrict__ planes, int *__restrict__ bad, double *__restrict__ dinv, int64_t o0,
                 int64_t o1, double *__restrict__ partials, double *__restrict__ planes64) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double g = 0.0;
    if (i < A.n) {
        float a[D];
        double a64[D];
#pragma unroll
        for (int s = 0; s < D; ++s) { a[s] = 0.0f; a64[s] = 0.0; }
        double diag = 1.0, sabs = 0.0;
        for (int32_t t = rowptr[i]; t < rowptr[i + 1]; ++t) {
            const int d = col[t] - (int)i;
            const double v64 = vals[t];
            const float v = (float)v64;
            sabs += fabs(v64);
            if (d == 0) diag = v64;
            bool hit = false;
#pragma unroll
            for (int s = 0; s < D; ++s)
                if (d == A.off[s]) {
                    a[s] = v;
                    a64[s] = v64;
                    hit = true;
                }
            if (!hit) *bad = 1;
        }
#pragma unroll
        for (int s = 0; s < D; ++s) planes[(int64_t)s * A.np + i] = a[s];
        if (planes64) {
#pragma unroll
            for (int s = 0; s < D; ++s) planes64[(int64_t)s * A.np + i] = a64[s];
        }
        const double di = (diag != 0.0) ? 1.0 / diag : 1.0;
        dinv[i] = di;
        planes[(int64_t)D * A.np + i] = (float)di;
        if (i >= o0 && i < o1) g = sabs * fabs(di);
    }
    __shared__ double sh[kThreads];
    sh[threadIdx.x] = g;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = sh[0];
}

enum DiaMode {
    DIA_PLAIN = 0,   // y = A x, or y = b - A x when b is given
    DIA_CHEB0 = 1,   // r = b - A x ; rout = r ; dout = c1 r / a_ii                     (first Chebyshev step, x untouched)
    DIA_CHEBK = 2,   // r = rin - A d ; [rout = r] ; dn = c1 d_i + c2 r / a_ii ; [dout = dn] ; xacc (+)= ... as SpmvEpi.xmode
    DIA_PRE2 = 3     // zero-guess degree-2 smoother: d0 = c0 b / a ; r = b - A d0 ; x = d0 + c1 d0 + c2 r / a_ii
};

struct DiaEpi {
    const double *b = nullptr, *rin = nullptr;
    double *rout = nullptr, *dout = nullptr, *xacc = nullptr;
    double c0 = 0.0, c1 = 0.0, c2 = 0.0;
    int xmode = 0;
    // rows this launch covers: [a0, a0+n0) then [a1, a1+n1); n0 < 0 = all rows.  Slab problems split every operator
    // application into the two lattice rows next to the ghost rows (launched behind the halo exchange on a second
    // stream) and the interior (launched at once, overlapping the exchange).
    int a0 = 0, n0 = -1, a1 = 0, n1 = 0;
};

// Row arithmetic of the V-cycle operator, shared by k_dia_apply and the fused level sweeps (mgsweep.cuh) so that both
// evaluate the same expression trees (same FMA contraction, same summation order => the same bits).
// acc = sum_s a_s xv_s as one fma chain, s = 0 .. D-1
// (a: the fp32 planes, or their exact fp64 conversions)
template <int D, class P>
__device__ __forceinline__ double dia_row_acc(const P *a, const double *xv) {
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < D; ++s) acc = fma((double)a[s], xv[s], acc);
    return acc;
}
// PRE2: xi = dinv_i b_i, acc = sum_s a_s dinv_j b_j ; d0 = c0 xi ; r = b_i - c0 acc ; x = d0 + c1 d0 + c2 dinv_i r
__device__ __forceinline__ double dia_pre2_row(double c0, double c1, double c2, double xi, double bi, double acc, double di) {
    const double d0i = c0 * xi;
    const double r = bi - c0 * acc;
    return d0i + c1 * d0i + c2 * di * r;
}
// PLAIN with a right-hand side: r = b_i - (A x)_i
__device__ __forceinline__ double dia_resid_row(double bi, double acc) { return bi - acc; }
// CHEB0: r = b_i - (A x)_i (returned) ; d = c1 dinv_i r
__device__ __forceinline__ double dia_cheb0_row(double c1, double bi, double acc, double di, double &d) {
    const double r = bi - acc;
    d = c1 * di * r;
    return r;
}
// CHEBK: r = rin_i - (A d)_i ; dn = c1 d_i + c2 dinv_i r (returned)
__device__ __forceinline__ double dia_chebk_row(double c1, double c2, double xi, double rin, double acc, double di, double &r) {
    r = rin - acc;
    return c1 * xi + c2 * di * r;
}

// One thread per row, 32-bit index arithmetic (int32 dofs), and an interior fast path without per-neighbour range
// checks (only the first and last w+1 rows of a lattice can reach outside [0,n)).  PRE2 gathers the scaled right-hand
// side c0 * dinv_j * b_j at the 7 neighbours from the dinv plane (no reciprocals, no staging).  PRE2 runs at 0.77 of
// the HBM peak where the other epilogues reach 0.95 - 1.00; ncu (profiles/r02_ncu_full_probe.csv) shows no saturated
// unit (DRAM 61 %, L2 40 %, L1 45 %, issue 39 %): the 14 gathers are consumed pairwise by their products, so a row
// exposes several memory round trips.  Two restructurings were measured and dropped (profiles/r02_summary.md): staging
// the gathers with 4 / 8-byte cp.async (211 us against 152 us) and a shared-memory tile of the three neighbour runs
// with coalesced loads (158 us).
template <int MODE, int D>
__global__ void __launch_bounds__(kThreads)
    k_dia_apply(DiaMat A, const double *__restrict__ x, double *__restrict__ y, DiaEpi E) {
    constexpr int SD = D / 2;           // the diagonal sits in the middle plane (offsets are symmetric about 0)
    const int n = (int)A.n;
    int i = blockIdx.x * kThreads + threadIdx.x;
    if (E.n0 >= 0) {                    // row selection (two segments)
        if (i >= E.n0 + E.n1) return;
        i = i < E.n0 ? E.a0 + i : E.a1 + (i - E.n0);
    }
    if (i >= n) return;
    const float *__restrict__ v = A.v + i;
    const size_t np = (size_t)A.np;
    float a[D];
#pragma unroll
    for (int s = 0; s < D; ++s) a[s] = __ldcs(v + s * np);
    const float *__restrict__ dinvp = A.v + (size_t)D * np;
    const double di = (MODE == DIA_PLAIN) ? 0.0 : (double)__ldcs(dinvp + i);      // Jacobi scaling 1/a_ii (not needed by the residual)
    const double *__restrict__ src = (MODE == DIA_PRE2) ? E.b : x;
    const bool interior = i + A.off[0] >= 0 && i + A.off[D - 1] < n;
    double xv[D];
    if (interior) {
#pragma unroll
        for (int s = 0; s < D; ++s) xv[s] = __ldg(src + (i + A.off[s]));
        if (MODE == DIA_PRE2) {
#pragma unroll
            for (int s = 0; s < D; ++s) xv[s] *= (s == SD) ? di : (double)__ldg(dinvp + (i + A.off[s]));
        }
    } else {
#pragma unroll
        for (int s = 0; s < D; ++s) {
            const int j = i + A.off[s];
            const bool ok = j >= 0 && j < n;
            xv[s] = ok ? __ldg(src + j) : 0.0;
            if (MODE == DIA_PRE2) xv[s] *= ok ? (double)__ldg(dinvp + j) : 0.0;
        }
    }
    const double acc = dia_row_acc<D>(a, xv), xi = xv[SD];
    if (MODE == DIA_PRE2) {             // xv = dinv_j b_j ; d0 = c0 xv ; r = b_i - A d0 ; x = d0 + c1 d0 + c2 dinv_i r
        y[i] = dia_pre2_row(E.c0, E.c1, E.c2, xi, __ldg(E.b + i), acc, di);
    } else if (MODE == DIA_PLAIN) {
        y[i] = E.b ? dia_resid_row(E.b[i], acc) : acc;
    } else if (MODE == DIA_CHEB0) {
        double d;
        E.rout[i] = dia_cheb0_row(E.c1, E.b[i], acc, di, d);
        E.dout[i] = d;
    } else {
        double r;
        const double dn = dia_chebk_row(E.c1, E.c2, xi, E.rin[i], acc, di, r);
        if (E.rout) E.rout[i] = r;
        if (E.dout) E.dout[i] = dn;
        if (E.xmode == 0) E.xacc[i] += dn;
        else if (E.xmode == 1) E.xacc[i] += xi + dn;
        else E.xacc[i] = xi + dn;
    }
}

// The Krylov recurrence's operator on fp64 planes (the exact assembled values, re-laid out): y = A x or y = b - A x,
// optionally with the fused partial sums of x_i y_i over the owned rows [o0,o1) (CG's p.Ap).  Persistent grid-stride
// kernel (bounded number of partials, fixed assignment => deterministic reduction).  76 bytes per row instead of the
// 104 of the CSR stream.
template <bool DOT, int D>
__global__ void __launch_bounds__(kThreads, 8)      // 8 CTAs per SM: the persistent grid (8 x SMs) must be resident in one wave
    k_dia_spmv64(const double *__restrict__ planes, DiaMat A, const double *__restrict__ x, double *__restrict__ y,
                 const double *__restrict__ b, int64_t o0, int64_t o1, double *__restrict__ partials, int a0, int n0, int a1,
                 int n1) {
    const int n = (int)A.n;
    const size_t np = (size_t)A.np;
    double dot = 0.0;
    const int total = n0 >= 0 ? n0 + n1 : n;
    for (int t = blockIdx.x * kThreads + threadIdx.x; t < total; t += gridDim.x * kThreads) {
        const int i = n0 < 0 ? t : (t < n0 ? a0 + t : a1 + (t - n0));
        double a[D];
#pragma unroll
        for (int s = 0; s < D; ++s) a[s] = __ldcs(planes + s * np + i);
        const bool interior = i + A.off[0] >= 0 && i + A.off[D - 1] < n;
        double acc = 0.0, xi = 0.0;
#pragma unroll
        for (int s = 0; s < D; ++s) {
            const int j = i + A.off[s];
            const double v = (interior || (j >= 0 && j < n)) ? __ldg(x + j) : 0.0;
            if (s == D / 2) xi = v;
            acc = fma(a[s], v, acc);
        }
        y[i] = b ? b[i] - acc : acc;
        if (DOT && i >= o0 && i < o1) dot += acc * xi;
    }
    if (DOT) {
        dot = block_sum(dot);
        if (threadIdx.x == 0) partials[blockIdx.x] = dot;
    }
}

}  // namespace femo
