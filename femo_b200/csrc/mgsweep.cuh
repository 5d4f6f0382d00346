// mgsweep.cuh -- one V-cycle visit of a large DIA lattice level in two stencil sweeps.
//
// The per-kernel visit of a fine level runs PRE2, PLAIN, k_restrict_nested, k_prolong_nested, CHEB0 and CHEBK: six
// passes over the level, 256 bytes per row, most of them intermediates (pre-smoothed x, r, prolonged x, the smoother's
// r and d) written to HBM and read back at once.  Here the level is visited twice:
//   down sweep  x_pre = PRE2(b) ; r = b - A x_pre ; rc = P^T r          reads b, 7 planes, dinv ; writes x_pre, rc
//   up sweep    x1 = x_pre + P xc ; r0, d0 = CHEB0(x1) ; x = CHEBK(d0)   reads x_pre, xc, b, planes, dinv ; writes x
// The offsets {-w-1, -w, -1, 0, 1, w, w+1} reach one node ring, so every stage needs its input on one more ring: a CTA
// owns a strip of `cols` lattice columns (+3 halo columns per side, one thread per column) and a band of coarse rows, and
// marches up the band row by row.  Rows move through small rings in shared memory; the values a thread only needs in its
// own column (planes, b, dinv) stay in registers.  Two barriers per row: the first stage's stencil reads rows written
// before the first, the second stage's reads the row the first stage has just written.  The planes are converted to
// fp64 once and serve both stencils (the conversions, not the FMAs, are the costly fp64-pipe work of a row).
//
// The row arithmetic is that of k_dia_apply / restrict_nested_at / prolong_nested_at (the shared helpers of stencil.cuh
// and multigrid.cuh), so the sweeps reproduce the per-kernel path bit for bit.  Positions off the lattice hold 0: the
// per-kernel path reads a wrapped neighbour there against a plane coefficient that is exactly 0 (k_csr_to_dia and the
// node-centric assembly store absent slots as 0.0f), and fma(0, v, acc) = acc for any finite v.
//
// x_pre goes to the level's work vector M.d (clobbered by the per-kernel post-smoother as well) and the up sweep writes
// the caller's x: a tile reads x on a halo ring that neighbouring CTAs own, so nothing is updated in place.
//
// Included by engine.cu after stencil.cuh, multigrid.cuh and mgfused.cuh.
#pragma once
#include "common.cuh"

namespace femo {

constexpr int kSwThreads = 256;                  // one thread per tile column
constexpr int kSwHalo = 3;                       // halo columns per side
constexpr int kSwMaxCols = kSwThreads - 2 * kSwHalo;
constexpr int kSwMinRows = 8;                    // coarse rows per CTA at least (the band's warm-up is 4 coarse rows)

struct SweepArgs {
    DiaMat A;                      // fine level: 7 fp32 planes + the fp32 Jacobi scaling plane
    int nx, ny;                    // fine cells per direction (even: 2:1 nested)
    int cols, rj;                  // owned lattice columns per strip (even), coarse rows per CTA
    const uint8_t *mask_f = nullptr, *mask_c = nullptr;
    double c0 = 0.0, c1 = 0.0, c2 = 0.0;   // down: PRE2 coefficients ; up: c0 = CHEB0's, c1 / c2 = CHEBK's
};

// fp32 -> fp64 (exact) kept as ONE conversion: left to itself the compiler sinks the conversion of a plane into each
// stencil that uses it and converts it twice per row
__device__ __forceinline__ double sw_f2d(float f) {
    double d;
    asm volatile("cvt.f64.f32 %0, %1;" : "=d"(d) : "f"(f));
    return d;
}

// stencil neighbours {-w-1, -w, -1, 0, 1, w, w+1} of column tx of row u from a row ring
template <int R, class T>
__device__ __forceinline__ void sw_gather(const T (*ring)[kSwThreads], int u, int tx, double (&xv)[7]) {
    const T *dn = ring[(u - 1) & (R - 1)], *md = ring[u & (R - 1)], *up = ring[(u + 1) & (R - 1)];
    xv[0] = dn[tx - 1]; xv[1] = dn[tx];
    xv[2] = md[tx - 1]; xv[3] = md[tx]; xv[4] = md[tx + 1];
    xv[5] = up[tx]; xv[6] = up[tx + 1];
}

__global__ void __launch_bounds__(kSwThreads, 4)
    k_mg_down(SweepArgs S, const double *__restrict__ b, double *__restrict__ xpre, double *__restrict__ rc) {
    __shared__ double sq[4][kSwThreads];     // dinv_j b_j (PRE2's scaled right-hand side)
    __shared__ double sx[4][kSwThreads];     // x_pre
    __shared__ double sr[4][kSwThreads];     // r = b - A x_pre (0 at Dirichlet nodes, as the restriction reads it)
    __shared__ double sb[8][kSwThreads];     // b, own column
    __shared__ float sdv[4][kSwThreads];     // dinv, own column
    const int tx = threadIdx.x;
    const int w = S.nx + 1, h = S.ny + 1, cw = S.nx / 2 + 1;
    const int c = blockIdx.x * S.cols - kSwHalo + tx;
    const bool colok = c >= 0 && c < w && tx < S.cols + 2 * kSwHalo;
    const bool inB = tx >= 1 && tx < S.cols + 2 * kSwHalo - 1, inC = tx >= 2 && tx < S.cols + 2 * kSwHalo - 2;
    const bool own = tx >= kSwHalo && tx < S.cols + kSwHalo;
    const int J0 = blockIdx.y * S.rj, J1 = min(J0 + S.rj, S.ny / 2 + 1);
    const int f0 = 2 * J0, f1 = min(2 * J1, h);                 // x_pre rows written by this CTA
    const size_t np = (size_t)S.A.np;
    const float *__restrict__ pl = S.A.v;
    const float *__restrict__ dvp = pl + 7 * np;
    // stage rows: A q at t in [2J0-3, 2J1+2] ; B x_pre at t-2 in [2J0-2, 2J1+1] ; C r at t-3 in [2J0-1, 2J1] ;
    // D rc of coarse row J at t = 2J+5
    const int t0 = 2 * J0 - 3, tend = 2 * J1 + 3;
    double nb = 0.0;
    float ndv = 0.0f, npl[7];
    auto loadA = [&](int t) {
        nb = 0.0;
        ndv = 0.0f;
        if (colok && t >= 0 && t < h && t <= 2 * J1 + 2) {
            const int k = t * w + c;
            nb = __ldg(b + k);
            ndv = __ldcs(dvp + k);
        }
    };
    auto loadB = [&](int u) {
#pragma unroll
        for (int s = 0; s < 7; ++s) npl[s] = 0.0f;
        if (colok && inB && u >= 0 && u < h && u >= 2 * J0 - 2 && u <= 2 * J1 + 1) {
            const int k = u * w + c;
#pragma unroll
            for (int s = 0; s < 7; ++s) npl[s] = __ldcs(pl + s * np + k);
        }
    };
    loadA(t0);
    loadB(t0 - 2);
    double pp[7];                              // fp64 planes of row t-3 (stage C), converted by stage B one row earlier
#pragma unroll
    for (int s = 0; s < 7; ++s) pp[s] = 0.0;
    for (int t = t0; t <= tend; ++t) {
        const double bt = nb;
        const float dvt = ndv;
        double pb[7];
#pragma unroll
        for (int s = 0; s < 7; ++s) pb[s] = sw_f2d(npl[s]);
        if (t < tend) {                        // next row's loads in flight while this row computes
            loadA(t + 1);
            loadB(t - 1);
        }
        __syncthreads();
        {   // A: q = dinv b on row t (0 off the lattice)
            const bool ok = colok && t >= 0 && t < h;
            sq[t & 3][tx] = ok ? bt * (double)dvt : 0.0;
            sb[t & 7][tx] = bt;
            sdv[t & 3][tx] = dvt;
        }
        {   // B: x_pre on row u = t-2
            const int u = t - 2;
            double xp = 0.0;
            if (colok && inB && u >= 0 && u < h && u >= 2 * J0 - 2 && u <= 2 * J1 + 1) {
                double xv[7];
                sw_gather<4>(sq, u, tx, xv);
                const double acc = dia_row_acc<7>(pb, xv);
                xp = dia_pre2_row(S.c0, S.c1, S.c2, xv[3], sb[u & 7][tx], acc, (double)sdv[u & 3][tx]);
                if (own && u >= f0 && u < f1) xpre[u * w + c] = xp;
            }
            sx[u & 3][tx] = xp;
        }
        __syncthreads();
        {   // C: r on row u = t-3
            const int u = t - 3;
            double r = 0.0;
            if (colok && inC && u >= 0 && u < h && u >= 2 * J0 - 1 && u <= 2 * J1) {
                double xv[7];
                sw_gather<4>(sx, u, tx, xv);
                r = dia_resid_row(sb[u & 7][tx], dia_row_acc<7>(pp, xv));
                if (S.mask_f && S.mask_f[u * w + c]) r = 0.0;
            }
            sr[u & 3][tx] = r;
        }
        {   // D: coarse row J = (t-5)/2 from r rows 2J-1 .. 2J+1 (written in earlier rows)
            const int J = (t - 5) >> 1;
            const int I = (blockIdx.x * S.cols + (tx - kSwHalo)) >> 1;
            if (!((t - 5) & 1) && J >= J0 && J < J1 && own && !((tx - kSwHalo) & 1) && I < cw) {
                const int j = 2 * J, q = J * cw + I;
                double v = 0.0;
                if (!(S.mask_c && S.mask_c[q]))
                    v = restrict_nested_val(sr[j & 3][tx], sr[j & 3][tx - 1], sr[j & 3][tx + 1], sr[(j - 1) & 3][tx],
                                            sr[(j + 1) & 3][tx], sr[(j - 1) & 3][tx - 1], sr[(j + 1) & 3][tx + 1]);
                rc[q] = v;
            }
        }
#pragma unroll
        for (int s = 0; s < 7; ++s) pp[s] = pb[s];
    }
}

__global__ void __launch_bounds__(kSwThreads, 3)
    k_mg_up(SweepArgs S, const double *__restrict__ b, const double *__restrict__ xpre, const double *__restrict__ xc,
            double *__restrict__ x) {
    __shared__ double sx1[8][kSwThreads];    // x1 = x_pre + P xc
    __shared__ double sd0[4][kSwThreads];    // d0 = c dinv r0
    __shared__ double sr0[4][kSwThreads];    // r0 = b - A x1, own column
    const int tx = threadIdx.x;
    const int w = S.nx + 1, h = S.ny + 1, cw = S.nx / 2 + 1;
    const int c = blockIdx.x * S.cols - kSwHalo + tx;
    const bool colok = c >= 0 && c < w && tx < S.cols + 2 * kSwHalo;
    const bool inA = tx >= 1 && tx < S.cols + 2 * kSwHalo - 1, inB = tx >= 2 && tx < S.cols + 2 * kSwHalo - 2;
    const bool own = tx >= kSwHalo && tx < S.cols + kSwHalo;
    const int J0 = blockIdx.y * S.rj, J1 = min(J0 + S.rj, S.ny / 2 + 1);
    const int f0 = 2 * J0, f1 = min(2 * J1, h);                 // x rows written by this CTA
    const size_t np = (size_t)S.A.np;
    const float *__restrict__ pl = S.A.v;
    // stage rows: A x1 at t in [f0-2, f1+1] ; B r0, d0 at t-2 in [f0-1, f1] ; C x at t-3 in [f0, f1)
    const int t0 = f0 - 2, tend = f1 + 2;
    double nxf = 0.0, na = 0.0, na2 = 0.0, nb = 0.0;
    bool nodd = false, nmask = false;
    float npl[8];
    auto loadA = [&](int t) {
        nxf = na = na2 = 0.0;
        nodd = nmask = false;
        if (colok && inA && t >= 0 && t < h && t <= f1 + 1) {
            const int k = t * w + c;
            nxf = __ldg(xpre + k);
            nmask = S.mask_f && S.mask_f[k];
            const int I = c >> 1, oi = c & 1, oj = t & 1, Jl = t >> 1;
            nodd = (oi | oj) != 0;
            if (!nmask) {
                na = __ldg(xc + Jl * cw + I);
                if (nodd) na2 = __ldg(xc + (Jl + oj) * cw + (I + oi));
            }
        }
    };
    auto loadB = [&](int u) {
        nb = 0.0;
#pragma unroll
        for (int s = 0; s < 8; ++s) npl[s] = 0.0f;
        if (colok && inB && u >= 0 && u < h && u >= f0 - 1 && u <= f1) {
            const int k = u * w + c;
#pragma unroll
            for (int s = 0; s < 8; ++s) npl[s] = __ldcs(pl + s * np + k);
            nb = __ldg(b + k);
        }
    };
    loadA(t0);
    loadB(t0 - 2);
    double pp[8];                              // fp64 planes + dinv of row t-3 (stage C), converted by stage B one row earlier
#pragma unroll
    for (int s = 0; s < 8; ++s) pp[s] = 0.0;
    for (int t = t0; t <= tend; ++t) {
        const double xf = nxf, a = na, a2 = na2, bu = nb;
        const bool odd = nodd, msk = nmask;
        double pb[8];
#pragma unroll
        for (int s = 0; s < 8; ++s) pb[s] = sw_f2d(npl[s]);
        if (t < tend) {
            loadA(t + 1);
            loadB(t - 1);
        }
        __syncthreads();
        {   // A: x1 on row t (Dirichlet nodes keep x_pre, as k_prolong_nested leaves them)
            double x1 = 0.0;
            if (colok && inA && t >= 0 && t < h) x1 = msk ? xf : prolong_nested_val(xf, a, a2, odd);
            sx1[t & 7][tx] = x1;
        }
        {   // B: r0 = b - A x1 ; d0 = c dinv r0 on row u = t-2
            const int u = t - 2;
            double r0 = 0.0, d0 = 0.0;
            if (colok && inB && u >= 0 && u < h && u >= f0 - 1 && u <= f1) {
                double xv[7];
                sw_gather<8>(sx1, u, tx, xv);
                r0 = dia_cheb0_row(S.c0, bu, dia_row_acc<7>(pb, xv), pb[7], d0);
            }
            sd0[u & 3][tx] = d0;
            sr0[u & 3][tx] = r0;
        }
        __syncthreads();
        {   // C: x = x1 + (d0 + d1) on row u = t-3
            const int u = t - 3;
            if (colok && own && u >= f0 && u < f1) {
                double xv[7], r;
                sw_gather<4>(sd0, u, tx, xv);
                const double dn = dia_chebk_row(S.c1, S.c2, xv[3], sr0[u & 3][tx], dia_row_acc<7>(pp, xv), pp[7], r);
                x[u * w + c] = sx1[u & 7][tx] + (xv[3] + dn);
            }
        }
#pragma unroll
        for (int s = 0; s < 8; ++s) pp[s] = pb[s];
    }
}

}  // namespace femo

using namespace femo;

// ---- host side -----------------------------------------------------------------------------------------------
// The sweeps take a level visit when the level is a single-GPU DIA lattice level with a 2:1 nested coarse level, the
// smoother is the fp32 degree-2 Chebyshev polynomial and the level is above the cooperative coarse kernel's range;
// FEMO_NO_MGSWEEP restores the per-kernel path (A/B switch).
static bool mgsweep_ok(const femo_problem *L, const femo_problem *C, const MgParams &mp) {
    return !g_env.no_mgsweep && mp.degree == 2 && level_op(L, mp.fp32) == LevelOp::DIA && nested_pair(L, C) &&
           !L->slab.active && !C->slab.active && !L->gpart.active && L->mgl.dia.nd == 7 &&
           L->state.ndofs > g_env.mgfused_max_rows;
}

// strips of near-equal even width, and bands of coarse rows sized so that the grid is about one wave of resident CTAs;
// the degree-2 Chebyshev coefficients (both sweeps use c0, c1, c2)
static int mgsweep_args(const femo_problem *L, const femo_problem *C, const void *kern, const MgParams &mp, SweepArgs &S,
                        dim3 &grid) {
    ChebPoly P(L->mgl.lmax, mp.ratio);
    P.next();
    S.c0 = P.c0; S.c1 = P.c1; S.c2 = P.c2;
    S.A = L->mgl.dia;
    S.nx = L->mesh.n[0];
    S.ny = L->mesh.n[1];
    S.mask_f = L->has_bc ? L->d_bc_mark : nullptr;
    S.mask_c = C->has_bc ? C->d_bc_mark : nullptr;
    const int w = S.nx + 1, ch = S.ny / 2 + 1;
    const int strips = (w + kSwMaxCols - 1) / kSwMaxCols;
    S.cols = ((w + strips - 1) / strips + 1) & ~1;
    int occ = 0;
    FEMO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSwThreads, 0));
    const int bands = std::max(1, std::max(1, occ) * L->num_sms / strips);
    S.rj = std::max(kSwMinRows, (ch + bands - 1) / bands);
    grid = dim3((unsigned)strips, (unsigned)((ch + S.rj - 1) / S.rj));
    return FEMO_OK;
}

// down sweep: x_pre = PRE2(b) into xpre, C->mgl.b = P^T (b - A x_pre)
static int mgsweep_down(femo_problem *L, femo_problem *C, const double *b, double *xpre, const MgParams &mp) {
    SweepArgs S;
    dim3 grid;
    int rc;
    if ((rc = mgsweep_args(L, C, (const void *)k_mg_down, mp, S, grid))) return rc;
    k_mg_down<<<grid, kSwThreads, 0, L->stream>>>(S, b, xpre, C->mgl.b);
    L->launches++;
    L->sweep_count[0]++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// up sweep: x = CHEBK(CHEB0(x_pre + P C->mgl.x)), the degree-2 post-smoother from the prolonged iterate
static int mgsweep_up(femo_problem *L, femo_problem *C, const double *b, const double *xpre, double *x, const MgParams &mp) {
    SweepArgs S;
    dim3 grid;
    int rc;
    if ((rc = mgsweep_args(L, C, (const void *)k_mg_up, mp, S, grid))) return rc;
    k_mg_up<<<grid, kSwThreads, 0, L->stream>>>(S, b, xpre, C->mgl.x, x);
    L->launches++;
    L->sweep_count[1]++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

static int mgsweep_vcycle(femo_problem *root, int lv, const double *b, double *x, const MgParams &mp, bool *done) {
    *done = false;
    femo_problem *L = mg_level(root, lv), *C = root->mg[lv];
    if (!mgsweep_ok(L, C, mp)) return FEMO_OK;
    int rc;
    if ((rc = mgsweep_down(L, C, b, L->mgl.d, mp))) return rc;
    if ((rc = mg_vcycle(root, lv + 1, C->mgl.b, C->mgl.x, mp))) return rc;
    if ((rc = mgsweep_up(L, C, b, L->mgl.d, x, mp))) return rc;
    *done = true;
    return FEMO_OK;
}
