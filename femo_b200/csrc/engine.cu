// engine.cu -- device kernels shared by all families (segmented reduction,
// boundary conditions, SpMV, fused Krylov vector kernels) and the C ABI.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "families.cuh"
#include "families2.cuh"
#include "families3.cuh"
#include "families4.cuh"
#include "families5.cuh"
#include "families6.cuh"
#include "families7.cuh"
#include "families8.cuh"
#include "lattice_asm.cuh"
#include "dist.cuh"

namespace femo {

thread_local std::string g_err;
EnvFlags g_env;
void refresh_env() {
    auto num = [](const char *name, long long dflt) { const char *e = getenv(name); return e ? atoll(e) : dflt; };
    g_env.no_dia = getenv("FEMO_NO_DIA") != nullptr;
    // BSR-3 is opt-in for the Krylov recurrence: measured on B200 (hexahedra, 6.5M dofs) 1.32 ms against 1.20 ms of the
    // CSR-stream kernel although it moves 29 % fewer bytes (latency-bound per block row; profiles/r02_summary.md)
    g_env.no_bsr = getenv("FEMO_BSR") == nullptr || getenv("FEMO_NO_BSR") != nullptr;
    g_env.no_overlap = getenv("FEMO_NO_OVERLAP") != nullptr;
    g_env.no_mgfused = getenv("FEMO_NO_MGFUSED") != nullptr;
    g_env.no_mgsweep = getenv("FEMO_NO_MGSWEEP") != nullptr;
    g_env.no_lattice_asm = getenv("FEMO_NO_LATTICE_ASM") != nullptr;
    g_env.no_graph = getenv("FEMO_NO_GRAPH") != nullptr;
    g_env.force_graph = getenv("FEMO_GRAPH") != nullptr;
    g_env.overlap_min_rows = num("FEMO_OVERLAP_MIN_ROWS", 1 << 20);
    g_env.mgfused_max_rows = num("FEMO_MGFUSED_MAX_ROWS", 20000);
    g_env.mgfused_ctas = num("FEMO_MGFUSED_CTAS", 0);
    g_env.mgfused_small_rows = num("FEMO_MGFUSED_SMALL_ROWS", 0);
    g_env.graph_max_rows = num("FEMO_GRAPH_MAX_ROWS", 1 << 20);
}
int set_err(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

// ===========================================================================
// sorted segmented reduction (K12): out[t] = sum_{s in [ptr[t],ptr[t+1])} scratch[src[s]]
// src is ascending inside every segment, so the summation order is fixed.
// ===========================================================================
__global__ void __launch_bounds__(kThreads) k_segreduce(const int32_t *__restrict__ ptr, const int32_t *__restrict__ src,
                                                        const double *__restrict__ scratch, double *__restrict__ out,
                                                        int64_t n) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int32_t s0 = ptr[t], s1 = ptr[t + 1];
    double acc = 0.0;
    for (int32_t s = s0; s < s1; ++s) acc += scratch[ld_stream(src + s)];
    out[t] = acc;
}

// Jacobian variant: one pass writes the un-BC'd values and/or the BC'd copy
// (rows and columns of Dirichlet dofs zeroed, diagonal = bc multiplicity;
// SURVEY.md Appendix A.2).  bcflag: 0 keep, 1 zero, 2 diagonal of a bc row.
__global__ void __launch_bounds__(kThreads)
    k_segreduce_jac(const int32_t *__restrict__ ptr, const int32_t *__restrict__ src, const double *__restrict__ scratch,
                    const uint8_t *__restrict__ bcflag, const int32_t *__restrict__ col,
                    const double *__restrict__ bc_diag, double *__restrict__ out, double *__restrict__ out_bc, int64_t n) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int32_t s0 = ptr[t], s1 = ptr[t + 1];
    double acc = 0.0;
    for (int32_t s = s0; s < s1; ++s) acc += scratch[ld_stream(src + s)];
    if (out) out[t] = acc;
    if (out_bc) {
        const uint8_t fl = bcflag ? bcflag[t] : 0;
        out_bc[t] = (fl == 0) ? acc : (fl == 1 ? 0.0 : bc_diag[col[t]]);
    }
}

// Uniform hexahedral lattices: every element matrix is rho_c^p times ONE unit-modulus block K0, so the Jacobian is
// reduced straight from (cell modulus, K0 entry) pairs -- the 4.6 KB per cell of element tensors never touch HBM.
// Same gather map, same summation order as the general path.
__global__ void __launch_bounds__(kThreads)
    k_segreduce_jac_k0(const int32_t *__restrict__ ptr, const int32_t *__restrict__ src, const double *__restrict__ k0,
                       const double *__restrict__ ec, uint32_t ne, const uint8_t *__restrict__ bcflag,
                       const int32_t *__restrict__ col, const double *__restrict__ bc_diag, double *__restrict__ out,
                       double *__restrict__ out_bc, int64_t n) {
    __shared__ double K[576];
    for (int t = threadIdx.x; t < 576; t += blockDim.x) K[t] = k0[t];
    __syncthreads();
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int32_t s0 = ptr[t], s1 = ptr[t + 1];
    double acc = 0.0;
    for (int32_t s = s0; s < s1; ++s) {
        const uint32_t q = (uint32_t)ld_stream(src + s);
        const uint32_t k = q / ne;
        acc += __ldg(ec + (q - k * ne)) * K[k];
    }
    if (out) out[t] = acc;
    if (out_bc) {
        const uint8_t fl = bcflag ? bcflag[t] : 0;
        out_bc[t] = (fl == 0) ? acc : (fl == 1 ? 0.0 : bc_diag[col[t]]);
    }
}

// NonlinearProblem.F boundary treatment (SURVEY.md A.4): for rows touching a
// Dirichlet column  b_i -= scale * sum_{j in bc} A_ij (g_j - x_j); then
// b[bc] = scale * (g - x).
__global__ void __launch_bounds__(kThreads)
    k_newton_rhs(const int32_t *__restrict__ rows, int64_t nrows, const int32_t *__restrict__ rowptr,
                 const int32_t *__restrict__ col, const double *__restrict__ vals, const uint8_t *__restrict__ mark,
                 const double *__restrict__ g, const double *__restrict__ x, double *__restrict__ b, double scale) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nrows) return;
    const int32_t i = rows[k];
    if (mark[i]) {
        b[i] = scale * (g[i] - (x ? x[i] : 0.0));
        return;
    }
    double acc = 0.0;
    for (int32_t t = rowptr[i]; t < rowptr[i + 1]; ++t) {
        const int32_t j = col[t];
        if (mark[j]) acc += vals[t] * (g[j] - (x ? x[j] : 0.0));
    }
    b[i] -= scale * acc;
}

// ===========================================================================
// reductions
// ===========================================================================
__global__ void __launch_bounds__(kThreads) k_sum(const double *__restrict__ a, int64_t n, double *__restrict__ partials) {
    double acc = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        acc += a[i];
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

__global__ void __launch_bounds__(kThreads)
    k_dot(const double *__restrict__ a, const double *__restrict__ b, int64_t n, double *__restrict__ partials) {
    double acc = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        acc += a[i] * b[i];
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// one CTA: fixed-order sum of np partials -> scalars[slot]
__global__ void __launch_bounds__(kThreads) k_finalize(const double *__restrict__ partials, int np, double *scalars, int slot) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < np; i += blockDim.x) acc += partials[i];
    acc = block_sum(acc);
    if (threadIdx.x == 0) scalars[slot] = acc;
}

// ===========================================================================
// SpMV (K7), CSR-stream: a CTA owns a block of consecutive rows whose nnz fit in
// shared memory.  Phase 1 streams values/columns of the whole block with fully
// coalesced, deeply unrolled loads (the addresses do not depend on the row
// structure, so many loads are in flight per thread) and stores val*x[col] in
// shared memory; phase 2 sums each row's products in a fixed order (one thread
// per row; the 7-9 entry rows of FE matrices give conflict-free strides) and
// writes y coalesced.  Optional fused dot(x, y) for CG.  Rows longer than the
// staging capacity are strided over by the whole CTA.
// ===========================================================================
// Row epilogues fused into the SpMV (applied by the thread that owns row i, acc = (A x)_i):
//   EPI_PLAIN   y_i = acc                      (or b_i - acc when b is given: residual)
//   EPI_CHEB0   r_i = b_i - acc ; d_i = c1 dinv_i r_i                      (first Chebyshev step, x untouched)
//   EPI_CHEBK   r_i = rin_i - acc ; dn = c1 x_i + c2 dinv_i r_i ; dout_i = dn   (x is the previous direction)
//               xacc_i: mode 0 += dn ; mode 1 += x_i + dn ; mode 2 = x_i + dn
enum SpmvEpiKind { EPI_PLAIN = 0, EPI_CHEB0 = 1, EPI_CHEBK = 2, EPI_ADD = 3 /* y_i += acc (prolongation x += P xc, amg.cuh) */ };
struct SpmvEpi {
    const double *b = nullptr, *dinv = nullptr, *rin = nullptr;
    double *rout = nullptr, *dout = nullptr, *xacc = nullptr;
    double c1 = 0.0, c2 = 0.0;
    int xmode = 0;
    int64_t own0 = 0, own1 = (int64_t)1 << 62;   // rows whose x_i*y_i enter the fused dot (owned dofs)
};

template <int EPI>
__device__ __forceinline__ void spmv_row_epilogue(const SpmvEpi &E, int64_t i, double acc, double xi, double *y) {
    if (EPI == EPI_PLAIN) {
        y[i] = E.b ? E.b[i] - acc : acc;
    } else if (EPI == EPI_ADD) {
        y[i] += acc;
    } else if (EPI == EPI_CHEB0) {
        const double r = E.b[i] - acc;
        E.rout[i] = r;
        E.dout[i] = E.c1 * E.dinv[i] * r;
    } else {
        const double r = E.rin[i] - acc;
        E.rout[i] = r;
        const double dn = E.c1 * xi + E.c2 * E.dinv[i] * r;
        E.dout[i] = dn;
        if (E.xmode == 0) E.xacc[i] += dn;
        else if (E.xmode == 1) E.xacc[i] += xi + dn;
        else E.xacc[i] = xi + dn;
    }
}

template <bool DOT, int EPI, class VT>
__global__ void __launch_bounds__(kThreads)
    k_spmv(const int32_t *__restrict__ rb, int nrb, const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
           const VT *__restrict__ vals, const double *__restrict__ x, double *__restrict__ y, SpmvEpi E,
           double *__restrict__ partials) {
    __shared__ double prod[kSpmvCap];
    __shared__ int32_t rp[kSpmvRows + 1];
    const int tid = threadIdx.x;
    double dot = 0.0;
    for (int blk = blockIdx.x; blk < nrb; blk += gridDim.x) {
        const int32_t r0 = rb[blk];
        const int nr = rb[blk + 1] - r0;
        for (int i = tid; i <= nr; i += kThreads) rp[i] = rowptr[r0 + i];
        __syncthreads();
        const int32_t s = rp[0], e = rp[nr];
        if (e - s <= kSpmvCap) {
            constexpr int U = 4;
            for (int32_t base = s + tid; base < e; base += kThreads * U) {
                int32_t c[U];
                double v[U];
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int32_t t = base + j * kThreads;
                    c[j] = (t < e) ? ld_stream(col + t) : 0;
                    v[j] = (t < e) ? ld_stream(vals + t) : 0.0;
                }
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int32_t t = base + j * kThreads;
                    if (t < e) prod[t - s] = v[j] * __ldg(x + c[j]);
                }
            }
            __syncthreads();
            if (e - s < 24 * nr) {             // short rows (P1 / Q1 scalar stencils): one thread per row
                for (int i = tid; i < nr; i += kThreads) {
                    double acc = 0.0;
                    for (int32_t k = rp[i] - s; k < rp[i + 1] - s; ++k) acc += prod[k];
                    const double xi = (DOT || EPI == EPI_CHEBK) ? __ldg(x + r0 + i) : 0.0;
                    spmv_row_epilogue<EPI>(E, r0 + i, acc, xi, y);
                    if (DOT && r0 + i >= E.own0 && r0 + i < E.own1) dot += acc * xi;
                }
            } else {                           // long rows (vector states in 3-D: 81 entries): 8 lanes per row,
                constexpr int L = 8;           // strided partial sums + fixed butterfly => still deterministic
                const int sub = tid & (L - 1);
                for (int base = 0; base < nr; base += kThreads / L) {
                    const int i = base + tid / L;
                    double acc = 0.0;
                    if (i < nr)
                        for (int32_t k = rp[i] - s + sub; k < rp[i + 1] - s; k += L) acc += prod[k];
#pragma unroll
                    for (int o = L / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                    if (sub == 0 && i < nr) {
                        const double xi = (DOT || EPI == EPI_CHEBK) ? __ldg(x + r0 + i) : 0.0;
                        spmv_row_epilogue<EPI>(E, r0 + i, acc, xi, y);
                        if (DOT && r0 + i >= E.own0 && r0 + i < E.own1) dot += acc * xi;
                    }
                }
            }
        } else {  // a single long row: CTA-wide strided reduction (fixed order)
            double acc = 0.0;
            for (int32_t t = s + tid; t < e; t += kThreads) acc += ld_stream(vals + t) * __ldg(x + ld_stream(col + t));
            acc = block_sum(acc);
            if (tid == 0) {
                const double xi = __ldg(x + r0);
                spmv_row_epilogue<EPI>(E, r0, acc, xi, y);
                if (DOT && r0 >= E.own0 && r0 < E.own1) dot += acc * xi;
            }
        }
        __syncthreads();
    }
    if (DOT) {
        dot = block_sum(dot);
        if (tid == 0) partials[blockIdx.x] = dot;
    }
}

__global__ void __launch_bounds__(kThreads)
    k_permute(const int32_t *__restrict__ perm, const double *__restrict__ in, double *__restrict__ out, int64_t n) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < n) out[t] = in[perm[t]];
}

// ===========================================================================
// BSR-3 SpMV (K7): vector states in 3-D couple nodes through complete 3x3 blocks, so one column index serves nine
// values: 72 + 4 bytes per block = 8.44 bytes per entry instead of the 12 of scalar CSR (SURVEY.md section 8d).
// Same CSR-stream scheme as k_spmv: a CTA owns consecutive block rows (<= kBsrBlocks blocks); phase 1 streams the
// block values coalesced into shared memory, phase 2 forms the three row-products of every block (one thread per
// (block, row)), phase 3 sums each scalar row over its blocks in a fixed order.  Optional fused dot(x, y).
// ===========================================================================
template <bool DOT>
__global__ void __launch_bounds__(kThreads)
    k_spmv_bsr3(int64_t nbrows, const int32_t *__restrict__ browptr, const int32_t *__restrict__ bcol,
                const double *__restrict__ bvals, const double *__restrict__ x, double *__restrict__ y,
                const double *__restrict__ bsub, int64_t own0, int64_t own1, double *__restrict__ partials) {
    // One warp per block row (3 scalar rows, ~27 blocks = 243 contiguous values): lanes stream the values of the block
    // row fully coalesced with 8 independent loads in flight, each value meets its x component (the three rows of a
    // block share the x triple through the cache), three accumulators per lane, fixed butterfly => deterministic.
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * kThreads) >> 5;
    double dot = 0.0;
    for (int64_t I = warp; I < nbrows; I += nwarps) {
        const int32_t s = __ldg(browptr + I), e = __ldg(browptr + I + 1);
        const double *v = bvals + (int64_t)s * 9;
        const int nv = (e - s) * 9;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        for (int t0 = 0; t0 < nv; t0 += 32 * 4) {
            double vv[4], xx[4];
            int rr[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = t0 + j * 32 + lane;
                vv[j] = 0.0; xx[j] = 0.0; rr[j] = 0;
                if (t < nv) {
                    const int k = t / 9, q = t - 9 * k;
                    rr[j] = q / 3;
                    vv[j] = ld_stream(v + t);
                    xx[j] = __ldg(x + 3 * (int64_t)__ldg(bcol + s + k) + (q - 3 * rr[j]));
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double pr = vv[j] * xx[j];
                a0 += rr[j] == 0 ? pr : 0.0;
                a1 += rr[j] == 1 ? pr : 0.0;
                a2 += rr[j] == 2 ? pr : 0.0;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a0 += __shfl_xor_sync(0xffffffffu, a0, o);
            a1 += __shfl_xor_sync(0xffffffffu, a1, o);
            a2 += __shfl_xor_sync(0xffffffffu, a2, o);
        }
        if (lane < 3) {
            const double acc = lane == 0 ? a0 : (lane == 1 ? a1 : a2);
            const int64_t row = 3 * I + lane;
            y[row] = bsub ? bsub[row] - acc : acc;
            if (DOT && row >= own0 && row < own1) dot += acc * __ldg(x + row);
        }
    }
    if (DOT) {
        dot = block_sum(dot);
        if (threadIdx.x == 0) partials[blockIdx.x] = dot;
    }
}

__global__ void __launch_bounds__(kThreads)
    k_diag_inv(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ vals,
               double *__restrict__ dinv, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double d = 1.0;
    for (int32_t t = rowptr[i]; t < rowptr[i + 1]; ++t)
        if (col[t] == i) d = vals[t];
    dinv[i] = (d != 0.0) ? 1.0 / d : 1.0;
}

__global__ void __launch_bounds__(kThreads) k_axpy(double a, const double *__restrict__ x, double *__restrict__ y, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] += a * x[i];
}

__global__ void __launch_bounds__(kThreads)
    k_divide(double a, const double *__restrict__ num, const double *__restrict__ den, double *__restrict__ out, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = a * num[i] / den[i];
}

// Cone density filter on the lattice of cell centres (examples/beam_topo_opt/pre_processor/
// general_filter_model.py:67-90): W_ij = (R - d_ij) / sum_k (R - d_ik) over centres with d <= R.
// The neighbour search is index arithmetic on the lattice (2-D: nz = 1); den_i = sum_k (R - d_ik) is geometry only.
struct FilterLat {
    int nx, ny, nz;
    double dx, dy, dz, R;
};

__global__ void __launch_bounds__(kThreads) k_filter_den(FilterLat L, double *__restrict__ den) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)L.nx * L.ny * L.nz) return;
    const int i = (int)(idx % L.nx), j = (int)((idx / L.nx) % L.ny), k = (int)(idx / ((int64_t)L.nx * L.ny));
    const int kx = (int)floor(L.R / L.dx), ky = (int)floor(L.R / L.dy), kz = L.nz > 1 ? (int)floor(L.R / L.dz) : 0;
    double s = 0.0;
    for (int c = max(k - kz, 0); c <= min(k + kz, L.nz - 1); ++c)
        for (int b = max(j - ky, 0); b <= min(j + ky, L.ny - 1); ++b)
            for (int a = max(i - kx, 0); a <= min(i + kx, L.nx - 1); ++a) {
                const double ex = (a - i) * L.dx, ey = (b - j) * L.dy, ez = (c - k) * L.dz;
                const double d = sqrt(ex * ex + ey * ey + ez * ez);
                if (d <= L.R) s += L.R - d;
            }
    den[idx] = s;
}

// out = W in (TRANSPOSE = false) or out = W^T in (true: weights normalised by the NEIGHBOUR's den)
template <bool TRANSPOSE>
__global__ void __launch_bounds__(kThreads)
    k_filter_apply(FilterLat L, const double *__restrict__ den, const double *__restrict__ in, double *__restrict__ out) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)L.nx * L.ny * L.nz) return;
    const int i = (int)(idx % L.nx), j = (int)((idx / L.nx) % L.ny), k = (int)(idx / ((int64_t)L.nx * L.ny));
    const int kx = (int)floor(L.R / L.dx), ky = (int)floor(L.R / L.dy), kz = L.nz > 1 ? (int)floor(L.R / L.dz) : 0;
    double s = 0.0;
    for (int c = max(k - kz, 0); c <= min(k + kz, L.nz - 1); ++c)
        for (int b = max(j - ky, 0); b <= min(j + ky, L.ny - 1); ++b)
            for (int a = max(i - kx, 0); a <= min(i + kx, L.nx - 1); ++a) {
                const double ex = (a - i) * L.dx, ey = (b - j) * L.dy, ez = (c - k) * L.dz;
                const double d = sqrt(ex * ex + ey * ey + ez * ez);
                if (d <= L.R) {
                    const int64_t q = ((int64_t)c * L.ny + b) * L.nx + a;
                    s += TRANSPOSE ? (L.R - d) * in[q] / den[q] : (L.R - d) * in[q];
                }
            }
    out[idx] = TRANSPOSE ? s : s / den[idx];
}

__global__ void __launch_bounds__(kThreads) k_fill(double a, double *__restrict__ y, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = a;
}

}  // namespace femo

using namespace femo;

// ===========================================================================
// helpers
// ===========================================================================
static inline int grid_for(int64_t n) { return (int)((n + kThreads - 1) / kThreads); }
static inline int red_grid(const femo_problem *p, int64_t n) {
    int64_t g = (n + kThreads - 1) / kThreads;
    int64_t cap = (int64_t)p->num_sms * 8;
    if (cap > kMaxPartials) cap = kMaxPartials;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, cap));
}

static int need_device(femo_problem *p) {
    if (!p) return set_err(FEMO_EINVAL, "null problem");
    refresh_env();
    if (!p->uploaded) return set_err(FEMO_ESTATE, "problem not uploaded to a CUDA device (femo_problem_upload); there is no CPU path");
    cudaError_t e = cudaSetDevice(p->device);
    if (e != cudaSuccess) return set_err(FEMO_ECUDA, cudaGetErrorString(e));
    return FEMO_OK;
}

static int need_coef(femo_problem *p, int slot, int64_t n, const char *what) {
    if (!p->coef[slot] || p->coefn[slot] != n)
        return set_err(FEMO_ESTATE, std::string("coefficient not set or wrong size: ") + what);
    return FEMO_OK;
}

static TriArgs tri_args(femo_problem *p, double *out) {
    TriArgs A;
    A.coords = p->d_coords;
    A.cellsT = p->d_cellsT;
    A.ncells = p->mesh.ncells;
    A.bf_cell = p->d_fb_cell;
    A.bf_local = p->d_fb_local;
    A.nfacets = (int64_t)p->fb_cell.size();
    A.u = p->coef[0];
    A.f = p->coef[1];
    A.uex = p->coef[2];
    A.alpha = p->params[0];
    A.beta = p->params[1];
    A.out = out;
    A.uex_tab = p->d_uex_tab;
    return A;
}

static BeamArgs beam_args(femo_problem *p, int out_id, double *out) {
    BeamArgs A;
    A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = p->mesh.ncells;
    A.fb_cell = p->d_fb_cell; A.fb_local = p->d_fb_local; A.nfacets = (int64_t)p->fb_cell.size();
    A.u = p->coef[0]; A.t = p->coef[1];
    A.E = p->params[0]; A.width = p->params[1]; A.L = p->params[2]; A.f = p->params[3];
    A.out_id = out_id; A.out = out;
    return A;
}

static QuadArgs quad_args(femo_problem *p, int out_id, double *out) {
    QuadArgs A;
    A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = p->mesh.ncells;
    A.fb_cell = p->d_fb_cell; A.fb_local = p->d_fb_local; A.nfacets = (int64_t)p->fb_cell.size();
    A.u = p->coef[0]; A.rho = p->coef[1];
    A.nu = p->params[0]; A.fx = p->params[1]; A.fy = p->params[2]; A.penal = p->params[3];
    A.volume = (p->mesh.hi[0] - p->mesh.lo[0]) * (p->mesh.hi[1] - p->mesh.lo[1]);
    A.out_id = out_id; A.out = out;
    return A;
}

static HexArgs hex_args(femo_problem *p, int out_id, double *out) {
    HexArgs A;
    A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = p->mesh.ncells;
    A.fb_cell = p->d_fb_cell; A.fb_local = p->d_fb_local; A.nfacets = (int64_t)p->fb_cell.size();
    A.u = p->coef[0]; A.rho = p->coef[1];
    A.nu = p->params[0]; A.f[0] = p->params[1]; A.f[1] = p->params[2]; A.f[2] = p->params[3]; A.penal = p->params[4];
    A.volume = (p->mesh.hi[0] - p->mesh.lo[0]) * (p->mesh.hi[1] - p->mesh.lo[1]) * (p->mesh.hi[2] - p->mesh.lo[2]);
    A.out_id = out_id; A.out = out;
    return A;
}

// the hexahedron cell kernel stages 32 cells' gradients in > 48 KB of dynamic shared memory
template <int OP>
static void launch_hex_cell(const HexArgs &A, cudaStream_t st) {
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(k_simp_hex_cell<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHexSmem);
        configured = true;
    }
    const int grid = (int)((A.ncells + kHexCells - 1) / kHexCells);
    k_simp_hex_cell<OP><<<grid, kThreads, kHexSmem, st>>>(A);
}

// unit-modulus 24x24 element matrix of an axis-aligned box cell (2x2x2 Gauss), local dof 3a+i, row-major
static void hex_unit_stiffness(double hx, double hy, double hz, double nu, std::vector<double> &K) {
    const double lam = nu / ((1.0 + nu) * (1.0 - 2.0 * nu)), mu = 1.0 / (2.0 * (1.0 + nu));
    const double g[2] = {0.5 - 0.28867513459481287, 0.5 + 0.28867513459481287}, h[3] = {hx, hy, hz};
    K.assign(576, 0.0);
    for (int q = 0; q < 8; ++q) {
        const double t[3] = {g[q & 1], g[(q >> 1) & 1], g[(q >> 2) & 1]};
        double G[8][3];
        for (int a = 0; a < 8; ++a) {
            const double l[3] = {(a & 1) ? t[0] : 1.0 - t[0], (a & 2) ? t[1] : 1.0 - t[1], (a & 4) ? t[2] : 1.0 - t[2]};
            G[a][0] = ((a & 1) ? 1.0 : -1.0) * l[1] * l[2] / h[0];
            G[a][1] = ((a & 2) ? 1.0 : -1.0) * l[0] * l[2] / h[1];
            G[a][2] = ((a & 4) ? 1.0 : -1.0) * l[0] * l[1] / h[2];
        }
        const double w = 0.125 * hx * hy * hz;
        for (int a = 0; a < 8; ++a)
            for (int b = 0; b < 8; ++b) {
                const double dot = G[a][0] * G[b][0] + G[a][1] * G[b][1] + G[a][2] * G[b][2];
                for (int i = 0; i < 3; ++i)
                    for (int j = 0; j < 3; ++j)
                        K[(3 * a + i) * 24 + 3 * b + j] += w * (lam * G[a][i] * G[b][j] + mu * G[a][j] * G[b][i] + (i == j ? mu * dot : 0.0));
            }
    }
}
static bool hex_matfree_level(const femo_problem *p) {
    return p->family == FEMO_FAMILY_SIMP_HEX8 && p->mesh.kind == MESH_HEX && p->mesh.lattice && !getenv("FEMO_NO_MATFREE");
}
// layout walk of a matrix-free level (lay_out_problem): K0 of its cells in the static arena, the cell moduli in the work arena
static void lay_out_matfree(femo_problem *L, Arena &st, Arena &wk) {
    if (!hex_matfree_level(L)) return;
    const Mesh &M = L->mesh;
    const double hx = (M.hi[0] - M.lo[0]) / M.n[0], hy = (M.hi[1] - M.lo[1]) / M.n[1];
    const double hz = (M.hi[2] - M.lo[2]) / (double)(L->slab.active ? L->slab.gny : M.n[2]);
    std::vector<double> K;
    hex_unit_stiffness(hx, hy, hz, L->params[0], K);
    put(st, L->mgl.k0, K);
    wk.take(L->mgl.ec, (size_t)M.ncells);
    if (!st.counting()) L->h_k0 = std::move(K);   // the moved buffer stays alive for the pending copy
}

// the analytic-u_ex table of THIS problem into constant memory, stream-ordered before the kernel that reads it
static int push_uex_table(femo_problem *p) {
    if (p->h_uex_tab.size() == 2 * 49 * 4)
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_uex49, p->h_uex_tab.data(), sizeof(double) * 2 * 49 * 4, 0, cudaMemcpyHostToDevice, p->stream));
    return FEMO_OK;
}

// number of scratch planes per entity of an op
static int op_planes(const femo_problem *p, int op) {
    const int nd = p->state.ndpc;
    switch (op) {
        case OP_RES: case OP_OUT_DU: return nd;
        case OP_JAC: return nd * nd;
        case OP_DRDM: return nd * p->in[0].ndpc;
        case OP_OUT_DM: return p->in[0].ndpc;
        default: return 1;
    }
}

// Run the element kernels of `op` (for output ops: of output `out_id`) over the blocks in
// `mask` into scratch: cells first, then the facet block at offset ncells*planes.
static int run_elements(femo_problem *p, int op, int mask, int out_id = 0) {
    const int64_t nc = p->mesh.ncells;
    const int64_t nf = (int64_t)p->fb_cell.size();
    cudaStream_t st = p->stream;
    int rc;
    if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
    const bool analytic_src = p->family == FEMO_FAMILY_MASS_P1 && p->params[1] < 1.5;
    const bool jac_reads_input = p->family == FEMO_FAMILY_SIMP_Q1 || p->family == FEMO_FAMILY_EB_BEAM ||
                                 p->family == FEMO_FAMILY_SIMP_HEX8 || p->family == FEMO_FAMILY_RM_PLATE ||
                                 p->family == FEMO_FAMILY_MOTOR_EM || p->family == FEMO_FAMILY_MOTOR_MM;
    if ((op != OP_JAC || jac_reads_input) && !analytic_src && (rc = need_coef(p, 1, p->in[0].ndofs, "input 0"))) return rc;
    double *cells_out = p->d_scratch;
    double *facets_out = p->d_scratch + ((mask & 1) ? nc * op_planes(p, op) : 0);
    const int gc = grid_for(nc), gf = grid_for(std::max<int64_t>(nf, 1));
#define FEMO_LAUNCH_OPS(KERNEL, GRID, ARGS)                                                   \
    switch (op) {                                                                             \
        case OP_RES: KERNEL<OP_RES><<<GRID, kThreads, 0, st>>>(ARGS); break;                  \
        case OP_JAC: KERNEL<OP_JAC><<<GRID, kThreads, 0, st>>>(ARGS); break;                  \
        case OP_DRDM: KERNEL<OP_DRDM><<<GRID, kThreads, 0, st>>>(ARGS); break;                \
        case OP_OUT: KERNEL<OP_OUT><<<GRID, kThreads, 0, st>>>(ARGS); break;                  \
        case OP_OUT_DU: KERNEL<OP_OUT_DU><<<GRID, kThreads, 0, st>>>(ARGS); break;            \
        case OP_OUT_DM: KERNEL<OP_OUT_DM><<<GRID, kThreads, 0, st>>>(ARGS); break;            \
    }                                                                                         \
    p->launches++;
    switch (p->family) {
        case FEMO_FAMILY_POISSON_P1: {
            if (op == OP_OUT || op == OP_OUT_DU)
                if ((rc = need_coef(p, 2, p->aux[0].ndofs, "u_ex"))) return rc;
            TriArgs A = tri_args(p, cells_out);
            FEMO_LAUNCH_OPS(k_poisson_p1_cell, gc, A)
            break;
        }
        case FEMO_FAMILY_NLPOISSON_P1: {
            if ((op == OP_OUT || op == OP_OUT_DU) && (rc = push_uex_table(p))) return rc;
            if (mask & 1) {
                TriArgs A = tri_args(p, cells_out);
                FEMO_LAUNCH_OPS(k_nlpoisson_p1_cell, gc, A)
            }
            if ((mask & 2) && nf > 0) {
                TriArgs F = tri_args(p, facets_out);
                if (op == OP_RES) k_nlpoisson_p1_facet<OP_RES><<<gf, kThreads, 0, st>>>(F);
                else k_nlpoisson_p1_facet<OP_JAC><<<gf, kThreads, 0, st>>>(F);
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_MOTOR_MM: {
            MmArgs A;
            A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = nc;
            A.fb_cell = p->d_fb_cell; A.fb_local = p->d_fb_local; A.nfacets = nf;
            A.tag = p->d_cell_tag; A.uh = p->coef[0]; A.g = p->coef[1];
            A.beta0 = p->params[0]; A.out_id = out_id;
            const int g1 = (int)((nc + 63) / 64), g2 = (int)((std::max<int64_t>(nf, 1) + 63) / 64);
            if (mask & 1) {
                A.out = cells_out;
                switch (op) {
                    case OP_RES: k_motor_mm<OP_RES, 0><<<g1, 64, 0, st>>>(A); break;
                    case OP_JAC: k_motor_mm<OP_JAC, 0><<<g1, 64, 0, st>>>(A); break;
                    case OP_OUT: k_motor_mm<OP_OUT, 0><<<g1, 64, 0, st>>>(A); break;
                    case OP_OUT_DU: k_motor_mm<OP_OUT_DU, 0><<<g1, 64, 0, st>>>(A); break;
                    default: return set_err(FEMO_EINVAL, "mesh-motion family: operation has no cell integral");
                }
                p->launches++;
            }
            if ((mask & 2) && nf > 0) {
                A.out = facets_out;
                if (op == OP_RES) k_motor_mm<OP_RES, 1><<<g2, 64, 0, st>>>(A);
                else if (op == OP_JAC) k_motor_mm<OP_JAC, 1><<<g2, 64, 0, st>>>(A);
                else if (op == OP_DRDM) k_motor_mm<OP_DRDM, 1><<<g2, 64, 0, st>>>(A);
                else return set_err(FEMO_EINVAL, "mesh-motion family: operation has no facet integral");
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_MOTOR_EM: {
            EmArgs A;
            A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = nc;
            A.fb_cell = p->d_fb_cell; A.fb_local = p->d_fb_local; A.nfacets = nf;
            A.tag = p->d_cell_tag; A.u = p->coef[0]; A.uh = p->coef[1];
            for (int k = 0; k < EM_NPARAM; ++k) A.prm[k] = p->params[k];
            A.out_id = out_id;
            const int g1 = (int)((nc + 127) / 128), g2 = (int)((std::max<int64_t>(nf, 1) + 127) / 128);
            if (mask & 1) {
                A.out = cells_out;
                switch (op) {
                    case OP_RES: k_motor_em<OP_RES, 0><<<g1, 128, 0, st>>>(A); break;
                    case OP_JAC: k_motor_em<OP_JAC, 0><<<g1, 128, 0, st>>>(A); break;
                    case OP_DRDM: k_motor_em<OP_DRDM, 0><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT: k_motor_em<OP_OUT, 0><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT_DU: k_motor_em<OP_OUT_DU, 0><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT_DM: k_motor_em<OP_OUT_DM, 0><<<g1, 128, 0, st>>>(A); break;
                }
                p->launches++;
            }
            if ((mask & 2) && nf > 0) {
                A.out = facets_out;
                if (op == OP_RES) k_motor_em<OP_RES, 1><<<g2, 128, 0, st>>>(A);
                else if (op == OP_JAC) k_motor_em<OP_JAC, 1><<<g2, 128, 0, st>>>(A);
                else k_motor_em<OP_DRDM, 1><<<g2, 128, 0, st>>>(A);
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_MASS_P1: {
            if (op != OP_RES && op != OP_JAC) return set_err(FEMO_EINVAL, "projection family: only residual and mass matrix");
            MassArgs A;
            A.coords = p->d_coords; A.cellsT = p->d_cellsT; A.ncells = nc;
            A.u = p->coef[0]; A.src = p->coef[1];
            A.target = (int)p->params[0]; A.source = (int)p->params[1]; A.power = p->params[2];
            A.out = cells_out;
            if (op == OP_RES) k_mass_cell<OP_RES><<<gc, kThreads, 0, st>>>(A);
            else k_mass_cell<OP_JAC><<<gc, kThreads, 0, st>>>(A);
            p->launches++;
            break;
        }
        case FEMO_FAMILY_EB_BEAM: {
            if (mask & 1) {
                BeamArgs A = beam_args(p, out_id, cells_out);
                FEMO_LAUNCH_OPS(k_beam_cell, gc, A)
            }
            if ((mask & 2) && nf > 0) {
                BeamArgs F = beam_args(p, out_id, facets_out);
                if (op == OP_RES) k_beam_facet<OP_RES><<<gf, kThreads, 0, st>>>(F);
                else if (op == OP_OUT) k_beam_facet<OP_OUT><<<gf, kThreads, 0, st>>>(F);
                else k_beam_facet<OP_OUT_DU><<<gf, kThreads, 0, st>>>(F);
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_SIMP_Q1: {
            if (mask & 1) {
                QuadArgs A = quad_args(p, out_id, cells_out);
                FEMO_LAUNCH_OPS(k_simp_q1_cell, gc, A)
            }
            if ((mask & 2) && nf > 0) {
                QuadArgs F = quad_args(p, out_id, facets_out);
                if (op == OP_RES) k_simp_q1_facet<OP_RES><<<gf, kThreads, 0, st>>>(F);
                else if (op == OP_OUT) k_simp_q1_facet<OP_OUT><<<gf, kThreads, 0, st>>>(F);
                else k_simp_q1_facet<OP_OUT_DU><<<gf, kThreads, 0, st>>>(F);
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_NLPOISSON_P2: {
            P2Args A;
            A.edgesT = p->d_edgesT;
            A.nverts = p->mesh.nverts;
            if (mask & 1) {
                A.T = tri_args(p, cells_out);
                FEMO_LAUNCH_OPS(k_nlpoisson_p2_cell, gc, A)
            }
            if ((mask & 2) && nf > 0) {
                A.T = tri_args(p, facets_out);
                if (op == OP_RES) k_nlpoisson_p2_facet<OP_RES><<<gf, kThreads, 0, st>>>(A);
                else k_nlpoisson_p2_facet<OP_JAC><<<gf, kThreads, 0, st>>>(A);
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_RM_PLATE: {
            if ((rc = need_coef(p, 2, p->in[1].ndofs, "input 1 (load)"))) return rc;
            RmArgs A;
            A.edgesT = p->d_edgesT;
            A.nverts = p->mesh.nverts; A.nedges = p->mesh.nedges;
            A.t = p->coef[1]; A.f = p->coef[2];
            A.E = p->params[0]; A.nu = p->params[1]; A.pen = p->params[2]; A.rho = p->params[3];
            A.out_id = out_id; A.slot = out_id;           // OP_DRDM: out_id carries the input slot
            const int g1 = (int)((nc + 127) / 128), g2 = (int)((std::max<int64_t>(nf, 1) + 127) / 128);
            if (mask & 1) {
                A.T = tri_args(p, cells_out);
                switch (op) {
                    case OP_RES: k_rm_plate_cell<OP_RES><<<g1, 128, 0, st>>>(A); break;
                    case OP_JAC: k_rm_plate_cell<OP_JAC><<<g1, 128, 0, st>>>(A); break;
                    case OP_DRDM: k_rm_plate_cell<OP_DRDM><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT: k_rm_plate_cell<OP_OUT><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT_DU: k_rm_plate_cell<OP_OUT_DU><<<g1, 128, 0, st>>>(A); break;
                    case OP_OUT_DM: k_rm_plate_cell<OP_OUT_DM><<<g1, 128, 0, st>>>(A); break;
                }
                p->launches++;
            }
            if ((mask & 2) && nf > 0) {
                A.T = tri_args(p, facets_out);
                if (op == OP_RES) k_rm_plate_facet<OP_RES><<<g2, 128, 0, st>>>(A);
                else if (op == OP_JAC) k_rm_plate_facet<OP_JAC><<<g2, 128, 0, st>>>(A);
                else return set_err(FEMO_EINVAL, "RM plate family: the penalty facets carry residual and Jacobian terms only");
                p->launches++;
            }
            break;
        }
        case FEMO_FAMILY_SIMP_HEX8: {
            if (mask & 1) {
                HexArgs A = hex_args(p, out_id, cells_out);
                switch (op) {
                    case OP_RES: launch_hex_cell<OP_RES>(A, st); break;
                    case OP_JAC: launch_hex_cell<OP_JAC>(A, st); break;
                    case OP_DRDM: launch_hex_cell<OP_DRDM>(A, st); break;
                    case OP_OUT: launch_hex_cell<OP_OUT>(A, st); break;
                    case OP_OUT_DM: launch_hex_cell<OP_OUT_DM>(A, st); break;
                    default: return set_err(FEMO_EINVAL, "hex SIMP family: no cell term for this operation");
                }
                p->launches++;
            }
            if ((mask & 2) && nf > 0) {
                HexArgs F = hex_args(p, out_id, facets_out);
                if (op == OP_RES) k_simp_hex_facet<OP_RES><<<gf, kThreads, 0, st>>>(F);
                else if (op == OP_OUT) k_simp_hex_facet<OP_OUT><<<gf, kThreads, 0, st>>>(F);
                else k_simp_hex_facet<OP_OUT_DU><<<gf, kThreads, 0, st>>>(F);
                p->launches++;
            }
            break;
        }
        default:
            return set_err(FEMO_EINVAL, "family has no device kernels in this build");
    }
#undef FEMO_LAUNCH_OPS
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

static int segreduce(femo_problem *p, const DevVecMap &m, int64_t n, double *d_out) {
    k_segreduce<<<grid_for(n), kThreads, 0, p->stream>>>(m.ptr, m.src, p->d_scratch, d_out, n);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

#include "dist_ops.cuh"

static inline int spmv_grid(const femo_problem *p, int nrb) {
    // persistent grid: every SM holds 8 CTAs and walks the row blocks with a grid stride, so the
    // rows in flight form one contiguous window (x stays L2-resident) and the dot partials are bounded
    int64_t cap = std::min<int64_t>((int64_t)p->num_sms * 8, kMaxPartials);
    return (int)std::max<int64_t>(1, std::min<int64_t>(nrb, cap));
}

template <bool DOT, class VT>
static int launch_spmv(femo_problem *p, const int32_t *rb, int nrb, const int32_t *rowptr, const int32_t *col,
                       const VT *vals, const double *x, double *y, const double *bsub, int *np_out,
                       bool halo = true) {
    // every SpMV on the state pattern refreshes the ghost rows of its input first (no-op on one GPU)
    if (halo) {
        int rc = halo_nodes(p, const_cast<double *>(x));
        if (rc) return rc;
    }
    const int grid = spmv_grid(p, nrb);
    SpmvEpi E;
    E.b = bsub;
    E.own0 = p->own_off;
    E.own1 = p->own_off + p->own_n;
    k_spmv<DOT, EPI_PLAIN, VT><<<grid, kThreads, 0, p->stream>>>(rb, nrb, rowptr, col, vals, x, y, E, p->d_partials);
    p->launches++;
    if (np_out) *np_out = grid;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// BSR-3 view of the dR/du values: re-layout once per solve, then every SpMV of the recurrence streams 8.44 B / entry
static inline bool bsr3_ready(const femo_problem *p) { return p->dpat[0].b_perm && p->d_bvals && !g_env.no_bsr; }
static int bsr3_convert(femo_problem *p, const double *vals) {
    const int64_t nnz = p->pat[0].nnz;
    k_permute<<<grid_for(nnz), kThreads, 0, p->stream>>>(p->dpat[0].b_perm, vals, p->d_bvals, nnz);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}
template <bool DOT>
static int launch_spmv_bsr3(femo_problem *p, const double *x, double *y, const double *bsub, int *np_out) {
    int rc = halo_nodes(p, const_cast<double *>(x));
    if (rc) return rc;
    const DevPattern &D = p->dpat[0];
    const int64_t nbrows = p->pat[0].nrows / 3;
    const int grid = spmv_grid(p, (int)std::min<int64_t>((nbrows + 7) / 8, 1 << 30));
    k_spmv_bsr3<DOT><<<grid, kThreads, 0, p->stream>>>(nbrows, D.b_rowptr, D.b_col, p->d_bvals, x, y, bsub, p->own_off,
                                                       p->own_off + p->own_n, p->d_partials);
    p->launches++;
    if (np_out) *np_out = grid;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// SpMV on pattern 0 with a fused Chebyshev epilogue (multigrid smoother)
template <class VT>
static int launch_spmv_cheb(femo_problem *p, int kind, const VT *vals, const double *x, const SpmvEpi &E) {
    const DevPattern &D = p->dpat[0];
    int rc = halo_nodes(p, const_cast<double *>(x));
    if (rc) return rc;
    const int grid = spmv_grid(p, D.nrb);
    if (kind == EPI_CHEB0)
        k_spmv<false, EPI_CHEB0, VT><<<grid, kThreads, 0, p->stream>>>(D.rb, D.nrb, D.rowptr, D.col, vals, x, nullptr, E, nullptr);
    else
        k_spmv<false, EPI_CHEBK, VT><<<grid, kThreads, 0, p->stream>>>(D.rb, D.nrb, D.rowptr, D.col, vals, x, nullptr, E, nullptr);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

static int read_scalars(femo_problem *p, int first, int count, double *h) {
    FEMO_CUDA(cudaMemcpyAsync(p->h_pinned, p->d_scalars + first, sizeof(double) * count, cudaMemcpyDeviceToHost, p->stream));
    FEMO_CUDA(cudaStreamSynchronize(p->stream));
    for (int i = 0; i < count; ++i) h[i] = p->h_pinned[i];
    return FEMO_OK;
}

// copy the Dirichlet arrays into their (always reserved) device slots
static int push_bc(femo_problem *p) {
    const int64_t N = p->state.ndofs;
    FEMO_CUDA(cudaSetDevice(p->device));
    if (p->bc_mark.empty()) {
        p->bc_mark.assign(N, 0);
        p->bc_g.assign(N, 0.0);
        p->bc_diag.assign(N, 0.0);
    }
    if (p->bcflag.empty()) p->bcflag.assign(p->pat[0].nnz, 0);
    cudaStream_t st = p->stream;
    FEMO_CUDA(cudaMemcpyAsync(p->d_bc_mark, p->bc_mark.data(), N, cudaMemcpyHostToDevice, st));
    FEMO_CUDA(cudaMemcpyAsync(p->d_bc_g, p->bc_g.data(), N * sizeof(double), cudaMemcpyHostToDevice, st));
    FEMO_CUDA(cudaMemcpyAsync(p->d_bc_diag, p->bc_diag.data(), N * sizeof(double), cudaMemcpyHostToDevice, st));
    FEMO_CUDA(cudaMemcpyAsync(p->dpat[0].bcflag, p->bcflag.data(), p->bcflag.size(), cudaMemcpyHostToDevice, st));
    if (!p->lift_rows.empty())
        FEMO_CUDA(cudaMemcpyAsync(p->d_lift_rows, p->lift_rows.data(), p->lift_rows.size() * sizeof(int32_t),
                                  cudaMemcpyHostToDevice, st));
    FEMO_CUDA(cudaStreamSynchronize(st));
    return FEMO_OK;
}

extern "C" {
static int propagate_bc(femo_problem *root, int start = 0);
static int set_bc_impl(femo_problem *p, const int32_t *dofs, const int32_t *list_ptr, int nlists, const double *g);
static int lattice_jacobian(femo_problem *p, double *d_vals, double *d_vals_bc, bool with_dia, bool dia_bc);
}

#include "stencil.cuh"
#include "multigrid.cuh"
#include "mgfused.cuh"
#include "mgsweep.cuh"
#include "amg.cuh"
#include "krylov.cuh"
#include "gmres.cuh"

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int femo_version(void) { return 100; }
const char *femo_last_error(void) { return g_err.c_str(); }

int femo_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---- meshes ---------------------------------------------------------------
int femo_mesh_create_unit_square(int nx, int ny, const double lo[2], const double hi[2], femo_mesh **out) {
    if (!out || nx < 1 || ny < 1 || !lo || !hi) return set_err(FEMO_EINVAL, "femo_mesh_create_unit_square: bad arguments");
    if ((int64_t)(nx + 1) * (ny + 1) > 2147483647LL) return set_err(FEMO_ELIMIT, "mesh exceeds int32 vertices");
    femo_mesh *m = new femo_mesh();
    make_unit_square_tri(nx, ny, lo, hi, m->m);
    *out = m;
    return FEMO_OK;
}
int femo_mesh_create_rectangle_quad(int nx, int ny, const double lo[2], const double hi[2], femo_mesh **out) {
    if (!out || nx < 1 || ny < 1 || !lo || !hi) return set_err(FEMO_EINVAL, "femo_mesh_create_rectangle_quad: bad arguments");
    femo_mesh *m = new femo_mesh();
    make_rectangle_quad(nx, ny, lo, hi, m->m);
    *out = m;
    return FEMO_OK;
}
int femo_mesh_create_box_hex(int nx, int ny, int nz, const double lo[3], const double hi[3], femo_mesh **out) {
    if (!out || nx < 1 || ny < 1 || nz < 1 || !lo || !hi) return set_err(FEMO_EINVAL, "femo_mesh_create_box_hex: bad arguments");
    if ((int64_t)(nx + 1) * (ny + 1) * (nz + 1) * 3 > 2147483647LL) return set_err(FEMO_ELIMIT, "mesh exceeds int32 dofs");
    femo_mesh *m = new femo_mesh();
    make_box_hex(nx, ny, nz, lo, hi, m->m);
    *out = m;
    return FEMO_OK;
}
int femo_mesh_create_from_arrays(int kind, int gdim, int64_t nverts, const double *coords, int64_t ncells, const int32_t *cells,
                                 femo_mesh **out) {
    if (!out || !coords || !cells) return set_err(FEMO_EINVAL, "femo_mesh_create_from_arrays: null");
    if (nverts * 3 > 2147483647LL || ncells > 2147483647LL) return set_err(FEMO_ELIMIT, "mesh exceeds int32");
    femo_mesh *m = new femo_mesh();
    try {
        make_from_arrays(kind, gdim, nverts, coords, ncells, cells, m->m);
    } catch (const LayoutError &e) {
        delete m;
        return set_err(e.code, e.msg);
    }
    *out = m;
    return FEMO_OK;
}
int femo_mesh_create_annulus(int nr, int nth, double r0, double r1, femo_mesh **out) {
    if (!out || nr < 1 || nth < 3 || !(r1 > r0) || !(r0 > 0)) return set_err(FEMO_EINVAL, "femo_mesh_create_annulus: bad arguments");
    femo_mesh *m = new femo_mesh();
    make_annulus_tri(nr, nth, r0, r1, m->m);
    *out = m;
    return FEMO_OK;
}

int femo_mesh_create_interval(int n, double x0, double x1, femo_mesh **out) {
    if (!out || n < 1) return set_err(FEMO_EINVAL, "femo_mesh_create_interval: bad arguments");
    femo_mesh *m = new femo_mesh();
    make_interval(n, x0, x1, m->m);
    *out = m;
    return FEMO_OK;
}
int femo_mesh_sizes(const femo_mesh *m, int64_t s[6]) {
    if (!m || !s) return set_err(FEMO_EINVAL, "femo_mesh_sizes: null");
    s[0] = m->m.ncells; s[1] = m->m.nverts; s[2] = m->m.nvpc; s[3] = m->m.gdim;
    s[4] = (int64_t)m->m.bf_cell.size(); s[5] = m->m.kind;
    return FEMO_OK;
}
int femo_mesh_copy(const femo_mesh *m, int what, void *out) {
    if (!m || !out) return set_err(FEMO_EINVAL, "femo_mesh_copy: null");
    const Mesh &M = m->m;
    switch (what) {
        case 0: memcpy(out, M.coords.data(), M.coords.size() * sizeof(double)); break;
        case 1: memcpy(out, M.cells.data(), M.cells.size() * sizeof(int32_t)); break;
        case 2: memcpy(out, M.bf_cell.data(), M.bf_cell.size() * sizeof(int32_t)); break;
        case 3: memcpy(out, M.bf_local.data(), M.bf_local.size() * sizeof(int32_t)); break;
        default: return set_err(FEMO_EINVAL, "femo_mesh_copy: bad selector");
    }
    return FEMO_OK;
}
void femo_mesh_destroy(femo_mesh *m) { delete m; }

// ---- problem layout -------------------------------------------------------
static int create_problem_impl(const Mesh &mesh, int family, const double *params, int nparams, bool jac_only,
                               const int32_t *tagged, int ntagged, femo_problem **out,
                               const int32_t *fcell = nullptr, const int32_t *flocal = nullptr, int nfl = 0,
                               const int32_t *cell_tags = nullptr) {
    femo_problem *p = new femo_problem();
    p->mesh = mesh;
    p->family = family;
    p->jac_only = jac_only;
    if (cell_tags) p->mesh.cell_tag.assign(cell_tags, cell_tags + mesh.ncells);
    for (int i = 0; i < nparams; ++i) p->params[i] = params[i];
    const Mesh &M = p->mesh;
    try {
        switch (family) {
            case FEMO_FAMILY_POISSON_P1:
            case FEMO_FAMILY_NLPOISSON_P1:
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                p->state.init(M, EL_VERTEX, 1);
                p->nin = 1;
                p->in[0].init(M, EL_DG0, 1);
                p->nout = 1;
                if (family == FEMO_FAMILY_POISSON_P1) {
                    p->naux = 1;  // u_ex in CG1 (run_poisson_opt.py:108)
                    p->aux[0].init(M, EL_VERTEX, 1);
                    if (nparams < 1) p->params[0] = 1e-6;
                } else {
                    p->res_mask = 3;
                    p->jac_mask = 3;
                    if (nparams < 1) p->params[0] = 6e-7;
                    if (nparams < 2) p->params[1] = 10.0;
                }
                break;
            case FEMO_FAMILY_MOTOR_MM:
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                if (M.cell_tag.empty()) throw LayoutError{FEMO_EINVAL, "motor family needs cell tags (subdomain ids)"};
                if (!fcell || !flocal) throw LayoutError{FEMO_EINVAL, "mesh-motion family needs the tagged one-sided facets dS(1000)/ds(1000)"};
                p->state.init(M, EL_VERTEX, 2);
                p->nin = 1;
                p->in[0].init(M, EL_VERTEX, 2);                 // prescribed edge displacement g = uhat_bc
                p->nout = 3;
                if (nparams < 1) p->params[0] = 5e3;
                p->res_mask = p->jac_mask = 3;
                p->drdm_mask = 2;                                // only the Nitsche facet terms depend on g
                for (int k = 0; k < 3; ++k) { p->out_mask[k] = 1; p->out_du_mask[k] = 1; p->out_dm_mask[k] = 0; }
                p->symmetric = false;
                break;
            case FEMO_FAMILY_MOTOR_EM:
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                if (M.cell_tag.empty()) throw LayoutError{FEMO_EINVAL, "motor family needs cell tags (subdomain ids)"};
                if (nparams < EM_NPARAM) throw LayoutError{FEMO_EINVAL, "motor family needs its full parameter vector"};
                p->state.init(M, EL_VERTEX, 1);
                p->nin = 1;
                p->in[0].init(M, EL_VERTEX, 2);                 // mesh displacement uhat
                p->nout = 2;
                p->res_mask = p->jac_mask = p->drdm_mask = 3;   // cells + exterior facets (Nitsche, Nanson normal)
                p->symmetric = false;                            // nonlinear Nitsche coefficient
                break;
            case FEMO_FAMILY_MASS_P1: {
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                const int target = (int)p->params[0], source = (int)p->params[1];
                p->state.init(M, target == 1 ? EL_DG0 : EL_VERTEX, 1);
                p->nin = 1;
                p->in[0].init(M, source == 3 ? EL_VERTEX : EL_DG0, 1);
                p->nout = 0;
                break;
            }
            case FEMO_FAMILY_EB_BEAM:
                if (M.kind != MESH_INTERVAL) throw LayoutError{FEMO_EINVAL, "family needs an interval mesh"};
                p->state.init(M, EL_HERMITE3, 2);
                p->nin = 1;
                p->in[0].init(M, EL_DG0, 1);
                p->nout = 2;
                if (nparams < 4) { p->params[0] = 1.0; p->params[1] = 0.1; p->params[2] = 1.0; p->params[3] = -1.0; }
                p->res_mask = 3;                               // cells + tip load ds(100)
                p->out_mask[0] = 2; p->out_du_mask[0] = 2; p->out_dm_mask[0] = 0;   // compliance
                p->out_mask[1] = 1; p->out_du_mask[1] = 0; p->out_dm_mask[1] = 1;   // volume
                break;
            case FEMO_FAMILY_SIMP_Q1:
                if (M.kind != MESH_QUAD) throw LayoutError{FEMO_EINVAL, "family needs a quadrilateral mesh"};
                p->state.init(M, EL_VERTEX, 2);
                p->nin = 1;
                p->in[0].init(M, EL_DG0, 1);
                p->nout = 2;
                if (nparams < 4) { p->params[0] = 0.3; p->params[1] = 0.0; p->params[2] = -0.25; p->params[3] = 3.0; }
                p->res_mask = 3;                               // cells + traction ds(100)
                p->out_mask[0] = 1; p->out_du_mask[0] = 0; p->out_dm_mask[0] = 1;   // average density
                p->out_mask[1] = 2; p->out_du_mask[1] = 2; p->out_dm_mask[1] = 0;   // compliance
                break;
            case FEMO_FAMILY_NLPOISSON_P2:
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                p->mesh.build_edges();
                p->state.init(M, EL_P2, 1);
                p->nin = 1;
                p->in[0].init(M, EL_DG0, 1);
                p->nout = 1;
                p->res_mask = 3;
                p->jac_mask = 3;
                if (nparams < 1) p->params[0] = 6e-7;
                if (nparams < 2) p->params[1] = 10.0;
                {   // vertex -> incident edges, ascending edge ids (restriction to the P1 multigrid level)
                    p->vptr.assign(M.nverts + 1, 0);
                    for (int64_t e = 0; e < M.nedges; ++e) { p->vptr[M.edge_verts[2 * e] + 1]++; p->vptr[M.edge_verts[2 * e + 1] + 1]++; }
                    for (int64_t v = 0; v < M.nverts; ++v) p->vptr[v + 1] += p->vptr[v];
                    p->vedge.resize(2 * M.nedges);
                    std::vector<int32_t> pos(p->vptr.begin(), p->vptr.end() - 1);
                    for (int64_t e = 0; e < M.nedges; ++e) { p->vedge[pos[M.edge_verts[2 * e]]++] = (int32_t)e; p->vedge[pos[M.edge_verts[2 * e + 1]]++] = (int32_t)e; }
                }
                break;
            case FEMO_FAMILY_RM_PLATE:
                if (M.kind != MESH_TRI) throw LayoutError{FEMO_EINVAL, "family needs a triangle mesh"};
                p->mesh.build_edges();
                p->state.init(M, EL_RMP, 1);
                p->nin = 2;
                p->in[0].init(M, EL_VERTEX, 1);                  // thickness (CG1)
                p->in[1].init(M, EL_VERTEX, 1);                  // transverse load (CG1)
                p->nout = 3;
                if (nparams < 4) { p->params[0] = 1.0e4; p->params[1] = 0.3; p->params[2] = 1.0e8; p->params[3] = 1.0; }   // E, nu, pen, rho
                p->res_mask = p->jac_mask = 3;                   // cells + penalty clamp on the facets of block 2
                p->drdm_mask = 1;
                p->out_mask[0] = 1; p->out_du_mask[0] = 1; p->out_dm_mask[0] = 0;   // compliance 1/2 int w^2
                p->out_mask[1] = 1; p->out_du_mask[1] = 0; p->out_dm_mask[1] = 1;   // mass
                p->out_mask[2] = 1; p->out_du_mask[2] = 1; p->out_dm_mask[2] = 1;   // elastic energy
                break;
            case FEMO_FAMILY_SIMP_HEX8:
                if (M.kind != MESH_HEX) throw LayoutError{FEMO_EINVAL, "family needs a hexahedral mesh"};
                p->state.init(M, EL_VERTEX, 3);
                p->nin = 1;
                p->in[0].init(M, EL_DG0, 1);
                p->nout = 2;
                if (nparams < 5) { p->params[0] = 0.3; p->params[1] = 0.0; p->params[2] = -0.25; p->params[3] = 0.0; p->params[4] = 3.0; }
                p->res_mask = 3;                               // cells + traction ds(100)
                p->out_mask[0] = 1; p->out_du_mask[0] = 0; p->out_dm_mask[0] = 1;   // average density
                p->out_mask[1] = 2; p->out_du_mask[1] = 2; p->out_dm_mask[1] = 0;   // compliance
                break;
            default:
                throw LayoutError{FEMO_EINVAL, "unknown form family"};
        }
        // block 2: all exterior facets (Nitsche) or the tagged subset (ds(tag) of the examples)
        if (fcell && flocal) {                       // explicit one-sided facets (cell, local facet)
            for (int k = 0; k < nfl; ++k) {
                if (fcell[k] < 0 || fcell[k] >= M.ncells || flocal[k] < 0 || flocal[k] >= (M.kind == MESH_HEX ? 6 : M.nvpc))
                    throw LayoutError{FEMO_EINVAL, "facet (cell, local) out of range"};
                p->fb_cell.push_back(fcell[k]);
                p->fb_local.push_back(flocal[k]);
            }
        } else if (family == FEMO_FAMILY_NLPOISSON_P1 || family == FEMO_FAMILY_NLPOISSON_P2 || family == FEMO_FAMILY_MOTOR_EM ||
                   (family == FEMO_FAMILY_RM_PLATE && !tagged)) {
            p->fb_cell = M.bf_cell;
            p->fb_local = M.bf_local;
        } else {
            for (int k = 0; k < ntagged; ++k) {
                if (tagged[k] < 0 || tagged[k] >= (int32_t)M.bf_cell.size())
                    throw LayoutError{FEMO_EINVAL, "tagged facet index out of range"};
                p->fb_cell.push_back(M.bf_cell[tagged[k]]);
                p->fb_local.push_back(M.bf_local[tagged[k]]);
            }
        }
        // node-centric Jacobian rows (lattice_asm.cuh): nonlinear Poisson P1 with Nitsche terms on ALL exterior facets
        p->lattice_fast = family == FEMO_FAMILY_NLPOISSON_P1 && M.lattice && M.kind == MESH_TRI && !fcell && p->jac_mask == 3;
        p->own_off = 0;
        p->own_n = p->state.ndofs;
        p->cown_off = 0;
        p->cown_n = M.ncells;
        IntegralBlock cells, facets;
        cells.ne = M.ncells;
        facets.ne = (int64_t)p->fb_cell.size();
        facets.ent_cell = p->fb_cell.data();
        p->blk[1] = {cells};
        p->blk[2] = {facets};
        p->blk[3] = {cells, facets};
        build_pattern(M, p->state, p->state, p->blk[p->jac_mask], p->pat[0]);
        if (!jac_only && p->state.element == EL_VERTEX && p->state.block == 3) build_bsr3(p->pat[0]);   // K7
        if (!jac_only) {  // coarse multigrid levels only ever assemble dR/du
            for (int s = 0; s < p->nin; ++s) build_pattern(M, p->state, p->in[s], p->blk[p->drdm_mask], p->pat[1 + s]);
            bool need[4] = {false, false, false, false};
            need[p->res_mask] = true;
            for (int k = 0; k < p->nout; ++k) need[p->out_du_mask[k]] = true;
            for (int m = 1; m < 4; ++m)
                if (need[m]) build_vecmap(M, p->state, p->blk[m], p->vm_state[m]);
            for (int s = 0; s < p->nin; ++s) build_vecmap(M, p->in[s], p->blk[1], p->vm_in[s]);
        }
    } catch (const LayoutError &e) {
        delete p;
        return set_err(e.code, e.msg);
    } catch (const std::exception &e) {
        delete p;
        return set_err(FEMO_EINVAL, e.what());
    }
    *out = p;
    return FEMO_OK;
}

int femo_problem_create(const femo_mesh *m, int family, const double *params, int nparams, femo_problem **out) {
    if (!m || !out) return set_err(FEMO_EINVAL, "femo_problem_create: null");
    if (nparams < 0 || nparams > 32) return set_err(FEMO_EINVAL, "femo_problem_create: nparams out of range");
    return create_problem_impl(m->m, family, params, nparams, false, nullptr, 0, out);
}

int femo_problem_create_ex(const femo_mesh *m, int family, const double *params, int nparams, const int32_t *facet_cell,
                           const int32_t *facet_local, int nfacets, const int32_t *cell_tags, femo_problem **out) {
    if (!m || !out || nfacets < 0) return set_err(FEMO_EINVAL, "femo_problem_create_ex: bad arguments");
    if (nparams < 0 || nparams > 32) return set_err(FEMO_EINVAL, "femo_problem_create_ex: nparams out of range");
    return create_problem_impl(m->m, family, params, nparams, false, nullptr, 0, out, facet_cell, facet_local, nfacets, cell_tags);
}

int femo_problem_set_param(femo_problem *p, int index, double value) {
    if (!p || index < 0 || index >= 32) return set_err(FEMO_EINVAL, "femo_problem_set_param: bad index");
    p->params[index] = value;
    for (femo_problem *c : p->mg) c->params[index] = value;
    return FEMO_OK;
}

int femo_problem_create_tagged(const femo_mesh *m, int family, const double *params, int nparams,
                               const int32_t *facet_ids, int nfacets, femo_problem **out) {
    if (!m || !out || nfacets < 0 || (nfacets > 0 && !facet_ids)) return set_err(FEMO_EINVAL, "femo_problem_create_tagged: bad arguments");
    if (nparams < 0 || nparams > 32) return set_err(FEMO_EINVAL, "femo_problem_create_tagged: nparams out of range");
    return create_problem_impl(m->m, family, params, nparams, false, facet_ids, nfacets, out);
}

// local problem of rank `rank` on its y-slab (one ghost cell row below, one ghost node row above)
static int create_slab_problem(int family, const double *params, int nparams, int nx, int gny, const double lo[2],
                               const double hi[2], int rank, int nranks, bool jac_only, femo_problem **out) {
    if (nranks < 1 || rank < 0 || rank >= nranks || gny % nranks != 0 || gny / nranks < 2)
        return set_err(FEMO_EINVAL, "slab partition needs gny divisible by the number of ranks and >= 2 rows per rank");
    SlabInfo sl = make_slab(gny, rank, nranks);
    Mesh m;
    make_unit_square_tri_slab(nx, gny, sl.crow0, sl.ncrows, lo, hi, m);
    int rc = create_problem_impl(m, family, params, nparams, jac_only, nullptr, 0, out);
    if (rc) return rc;
    femo_problem *p = *out;
    p->slab = sl;
    const int64_t row_len = (int64_t)(nx + 1) * p->state.block, crow_len = m.ncells / sl.ncrows;
    p->own_off = sl.own0 * row_len;
    p->own_n = (int64_t)(sl.own1 - sl.own0) * row_len;
    p->cown_off = sl.cown0 * crow_len;
    p->cown_n = (int64_t)(sl.cown1 - sl.cown0) * crow_len;
    return FEMO_OK;
}

// local problem of rank `rank` on its z-slab of the hexahedral box; `face_mask` bit l tags every exterior facet with
// local facet id l (0 z=lo, 1 y=lo, 2 x=lo, 3 x=hi, 4 y=hi, 5 z=hi) as a traction facet ds(100)
static int create_slab_problem_hex(int family, const double *params, int nparams, int nx, int ny, int gnz, const double lo[3],
                                   const double hi[3], int rank, int nranks, bool jac_only, int face_mask, femo_problem **out) {
    if (nranks < 1 || rank < 0 || rank >= nranks || gnz % nranks != 0 || gnz / nranks < 2)
        return set_err(FEMO_EINVAL, "slab partition needs gnz divisible by the number of ranks and >= 2 layers per rank");
    SlabInfo sl = make_slab(gnz, rank, nranks);
    Mesh m;
    make_box_hex_slab(nx, ny, gnz, sl.crow0, sl.ncrows, lo, hi, m);
    std::vector<int32_t> tagged;
    for (size_t k = 0; k < m.bf_local.size(); ++k)
        if ((face_mask >> m.bf_local[k]) & 1) tagged.push_back((int32_t)k);
    int rc = create_problem_impl(m, family, params, nparams, jac_only, tagged.data(), (int)tagged.size(), out);
    if (rc) return rc;
    femo_problem *p = *out;
    p->slab = sl;
    const int64_t row_len = (int64_t)(nx + 1) * (ny + 1) * p->state.block, crow_len = (int64_t)nx * ny;
    p->own_off = sl.own0 * row_len;
    p->own_n = (int64_t)(sl.own1 - sl.own0) * row_len;
    p->cown_off = sl.cown0 * crow_len;
    p->cown_n = (int64_t)(sl.cown1 - sl.cown0) * crow_len;
    p->fown_off = 0;
    while (p->fown_off < (int64_t)p->fb_cell.size() && p->fb_cell[p->fown_off] < p->cown_off) p->fown_off++;
    p->face_mask = face_mask;
    return FEMO_OK;
}

int femo_problem_create_slab_hex(int family, const double *params, int nparams, int nx, int ny, int gnz, const double lo[3],
                                 const double hi[3], int rank, int nranks, int face_mask, femo_problem **out) {
    if (!out || !lo || !hi || nx < 1 || ny < 1 || nparams < 0 || nparams > 8)
        return set_err(FEMO_EINVAL, "femo_problem_create_slab_hex: bad arguments");
    if (family != FEMO_FAMILY_SIMP_HEX8) return set_err(FEMO_EINVAL, "z-slab partitioning is available for the hexahedral SIMP family");
    return create_slab_problem_hex(family, params, nparams, nx, ny, gnz, lo, hi, rank, nranks, false, face_mask, out);
}

int femo_problem_create_slab(int family, const double *params, int nparams, int nx, int gny, const double lo[2],
                             const double hi[2], int rank, int nranks, femo_problem **out) {
    if (!out || !lo || !hi || nx < 1 || nparams < 0 || nparams > 8) return set_err(FEMO_EINVAL, "femo_problem_create_slab: bad arguments");
    if (family != FEMO_FAMILY_POISSON_P1 && family != FEMO_FAMILY_NLPOISSON_P1)
        return set_err(FEMO_EINVAL, "slab partitioning is available for the P1 triangle families");
    return create_slab_problem(family, params, nparams, nx, gny, lo, hi, rank, nranks, false, out);
}

int femo_problem_mesh_sizes(const femo_problem *p, int64_t s[6]) {
    if (!p || !s) return set_err(FEMO_EINVAL, "femo_problem_mesh_sizes: null");
    s[0] = p->mesh.ncells; s[1] = p->mesh.nverts; s[2] = p->mesh.nvpc; s[3] = p->mesh.gdim;
    s[4] = (int64_t)p->mesh.bf_cell.size(); s[5] = p->mesh.kind;
    return FEMO_OK;
}

int femo_problem_mesh_copy(const femo_problem *p, int what, void *out) {
    if (!p || !out) return set_err(FEMO_EINVAL, "femo_problem_mesh_copy: null");
    femo_mesh tmp;
    const Mesh &M = p->mesh;
    switch (what) {
        case 0: memcpy(out, M.coords.data(), M.coords.size() * sizeof(double)); break;
        case 1: memcpy(out, M.cells.data(), M.cells.size() * sizeof(int32_t)); break;
        case 2: memcpy(out, M.bf_cell.data(), M.bf_cell.size() * sizeof(int32_t)); break;
        case 3: memcpy(out, M.bf_local.data(), M.bf_local.size() * sizeof(int32_t)); break;
        case 4: memcpy(out, M.edge_verts.data(), M.edge_verts.size() * sizeof(int32_t)); break;   // P2: (nedges,2)
        case 5: memcpy(out, M.cell_edges.data(), M.cell_edges.size() * sizeof(int32_t)); break;   // P2: (ncells,3)
        default: return set_err(FEMO_EINVAL, "femo_problem_mesh_copy: bad selector");
    }
    (void)tmp;
    return FEMO_OK;
}

int femo_problem_slab_info(const femo_problem *p, int64_t info[16]) {
    if (!p || !info) return set_err(FEMO_EINVAL, "femo_problem_slab_info: null");
    const SlabInfo &s = p->slab;
    const int64_t v[13] = {s.active, s.rank, s.nranks, s.gny, s.crow0, s.ncrows, s.own0, s.own1, s.cown0, s.cown1,
                           p->own_off, p->own_n, p->cown_off};
    for (int i = 0; i < 13; ++i) info[i] = v[i];
    info[13] = p->cown_n; info[14] = p->mesh.n[0]; info[15] = p->mesh.n[1];
    return FEMO_OK;
}

// Distributed multigrid levels keep at least this many lattice rows per rank; coarser levels are replicated
// (their work is < 1% of the fine level, and every distributed level costs ~5 halo exchanges per V-cycle).
// FEMO_DIST_MIN_ROWS overrides (the tests use 16 to exercise several distributed levels on small meshes).
static int dist_min_rows() {
    const char *e = getenv("FEMO_DIST_MIN_ROWS");
    int v = e ? atoi(e) : 128;
    return v < 2 ? 2 : v;
}

static int enable_multigrid_slab_hex(femo_problem *p) {
    int nx = p->mesh.n[0], ny = p->mesh.n[1], gnz = p->slab.gny;
    const int R = p->slab.nranks, rank = p->slab.rank;
    int rows = gnz / R, rc;
    const int kDistMinRows = std::max(2, dist_min_rows() / 8);     // a z-layer holds a whole plane of nodes
    // one more distributed level only if a 2:1 nested replicated level still fits below it
    while (rows % 4 == 0 && nx % 4 == 0 && ny % 4 == 0 && rows / 2 >= kDistMinRows) {
        nx /= 2; ny /= 2; gnz /= 2; rows /= 2;
        femo_problem *c = nullptr;
        if ((rc = create_slab_problem_hex(p->family, p->params, 32, nx, ny, gnz, p->mesh.lo, p->mesh.hi, rank, R, true, 0, &c))) return rc;
        c->parent = p;
        p->mg.push_back(c);
    }
    if (rows % 2 != 0 || nx % 2 != 0 || ny % 2 != 0)
        return set_err(FEMO_EINVAL, "partitioned multigrid needs nx, ny and layers-per-rank divisible by 2 down to the replicated level (use powers of two)");
    nx /= 2; ny /= 2; gnz /= 2;                                  // replicated levels: the whole coarse box on every rank
    bool first = true;
    while (first || nx > 4 || ny > 4 || gnz > 4 || (int64_t)(nx + 1) * (ny + 1) * (gnz + 1) * 3 > kMgDenseMax) {
        if (!first) {
            if (nx == 1 && ny == 1 && gnz == 1) break;
            nx = std::max(1, (nx + 1) / 2); ny = std::max(1, (ny + 1) / 2); gnz = std::max(1, (gnz + 1) / 2);
        }
        first = false;
        Mesh cm;
        make_box_hex(nx, ny, gnz, p->mesh.lo, p->mesh.hi, cm);
        femo_problem *c = nullptr;
        if ((rc = create_problem_impl(cm, p->family, p->params, 32, true, nullptr, 0, &c))) return rc;
        c->parent = p;
        c->replicated = true;
        p->mg.push_back(c);
    }
    if (!p->bc_mark.empty()) return propagate_bc(p);
    return FEMO_OK;
}

static int enable_multigrid_slab(femo_problem *p) {
    if (p->mesh.kind == MESH_HEX) return enable_multigrid_slab_hex(p);
    int nx = p->mesh.n[0], gny = p->slab.gny;
    const int R = p->slab.nranks, rank = p->slab.rank;
    int rows = gny / R, rc;
    // A distributed level costs ~5 neighbour synchronisations per V-cycle (about 13 us each, measured on 2 B200s:
    // profiles/r02_summary.md), a replicated one costs its redundant arithmetic on every rank: levels stay distributed
    // while their global lattice has more than ~600k nodes (FEMO_DIST_MIN_ROWS fixes the cut instead).
    const bool fixed_cut = getenv("FEMO_DIST_MIN_ROWS") != nullptr;
    const int kDistMinRows = fixed_cut ? dist_min_rows() : 2;
    auto keep_distributed = [&](int cnx, int cgny) { return fixed_cut || (int64_t)(cnx + 1) * (cgny + 1) > 600000; };
    while (rows % 2 == 0 && nx % 2 == 0 && rows / 2 >= kDistMinRows && nx / 2 >= 2 && (rows / 2) % 2 == 0 && (nx / 2) % 2 == 0 &&
           keep_distributed(nx / 2, gny / 2)) {
        nx /= 2; gny /= 2; rows /= 2;
        femo_problem *c = nullptr;
        if ((rc = create_slab_problem(p->family, p->params, 32, nx, gny, p->mesh.lo, p->mesh.hi, rank, R, true, &c))) return rc;
        c->parent = p;
        p->mg.push_back(c);
    }
    if (rows % 2 != 0 || nx % 2 != 0)
        return set_err(FEMO_EINVAL, "partitioned multigrid needs nx and rows-per-rank divisible by 2 down to the replicated level (use powers of two)");
    // replicated levels: the whole coarse lattice on every rank
    nx /= 2; gny /= 2;
    bool first = true;
    while (first || nx > kMgCoarsest || gny > kMgCoarsest) {
        if (!first) {
            if (nx > kMgCoarsest) nx = (nx + 1) / 2;
            if (gny > kMgCoarsest) gny = (gny + 1) / 2;
        }
        first = false;
        Mesh cm;
        make_unit_square_tri(nx, gny, p->mesh.lo, p->mesh.hi, cm);
        femo_problem *c = nullptr;
        if ((rc = create_problem_impl(cm, p->family, p->params, 32, true, nullptr, 0, &c))) return rc;
        c->parent = p;
        c->replicated = true;
        p->mg.push_back(c);
    }
    if (!p->bc_mark.empty()) return propagate_bc(p);
    return FEMO_OK;
}

int femo_problem_enable_multigrid(femo_problem *p) {
    if (!p) return set_err(FEMO_EINVAL, "femo_problem_enable_multigrid: null");
    if (p->uploaded) return set_err(FEMO_ESTATE, "femo_problem_enable_multigrid must precede femo_problem_upload");
    if (!p->mesh.lattice) return set_err(FEMO_EINVAL, "multigrid needs a lattice mesh");
    const bool tri = p->mesh.kind == MESH_TRI && p->state.element == EL_VERTEX && p->state.block == 1;
    const bool quad = p->mesh.kind == MESH_QUAD && p->state.element == EL_VERTEX;
    const bool hex = p->mesh.kind == MESH_HEX && p->state.element == EL_VERTEX;
    const bool p2 = p->mesh.kind == MESH_TRI && p->state.element == EL_P2 && !p->slab.active;
    if (!tri && !quad && !hex && !p2)
        return set_err(FEMO_EINVAL, "multigrid is available for vertex-based states on lattice triangle / quadrilateral / hexahedral meshes");
    if (!p->mg.empty()) return FEMO_OK;
    if (p->slab.active) return enable_multigrid_slab(p);
    int nx = p->mesh.n[0], ny = p->mesh.n[1], nz = p->mesh.n[2];
    // P2: the first coarse level is the P1 family on the SAME mesh (p-multigrid), then the lattice is coarsened
    const int child_family = p2 ? FEMO_FAMILY_NLPOISSON_P1 : p->family;
    if (p2) {
        Mesh cm;
        make_unit_square_tri(nx, ny, p->mesh.lo, p->mesh.hi, cm);
        femo_problem *c = nullptr;
        int rc = create_problem_impl(cm, child_family, p->params, 32, true, nullptr, 0, &c);
        if (rc) return rc;
        c->parent = p;
        p->mg.push_back(c);
    }
    // coarsen until the coarsest system fits the explicit inverse (<= 512 dofs)
    const int coarsest = hex ? 4 : ((p->state.block > 1) ? 6 : kMgCoarsest);
    while (nx > coarsest || ny > coarsest || nz > coarsest ||
           (hex && (int64_t)(nx + 1) * (ny + 1) * (nz + 1) * p->state.block > kMgDenseMax)) {
        if (hex) {   // halve every direction that still can be
            if (nx == 1 && ny == 1 && nz == 1) break;
            nx = std::max(1, (nx + 1) / 2);
            ny = std::max(1, (ny + 1) / 2);
            nz = std::max(1, (nz + 1) / 2);
        } else {
            if (nx > coarsest) nx = (nx + 1) / 2;
            if (ny > coarsest) ny = (ny + 1) / 2;
        }
        Mesh cm;
        if (hex) make_box_hex(nx, ny, nz, p->mesh.lo, p->mesh.hi, cm);
        else if (quad) make_rectangle_quad(nx, ny, p->mesh.lo, p->mesh.hi, cm);
        else make_unit_square_tri(nx, ny, p->mesh.lo, p->mesh.hi, cm);
        femo_problem *c = nullptr;
        int rc = create_problem_impl(cm, child_family, p->params, 32, true, nullptr, 0, &c);
        if (rc) return rc;
        c->parent = p;
        p->mg.push_back(c);
    }
    if (!p->bc_mark.empty()) return propagate_bc(p);
    return FEMO_OK;
}

int femo_problem_mg_levels(const femo_problem *p) { return p ? (int)p->mg.size() + 1 : 0; }

void femo_problem_destroy(femo_problem *p) {
    if (!p) return;
    for (femo_problem *c : p->mg) femo_problem_destroy(c);
    delete p->amg;
    if (p->h_pinned) cudaFreeHost(p->h_pinned);
    if (!p->parent && p->stream2) {
        cudaStreamDestroy(p->stream2);
        cudaEventDestroy(p->ev_fork);
        cudaEventDestroy(p->ev_join);
    }
    delete p;
}

int femo_problem_sizes(const femo_problem *p, int64_t s[16]) {
    if (!p || !s) return set_err(FEMO_EINVAL, "femo_problem_sizes: null");
    for (int i = 0; i < 16; ++i) s[i] = 0;
    s[0] = p->state.ndofs; s[1] = p->nin; s[2] = p->naux; s[3] = p->nout;
    for (int i = 0; i < p->nin; ++i) s[4 + i] = p->in[i].ndofs;
    for (int i = 0; i < p->naux; ++i) s[8 + i] = p->aux[i].ndofs;
    s[12] = (int64_t)p->fb_cell.size();
    return FEMO_OK;
}

static const Pattern *get_pat(const femo_problem *p, int which) {
    if (!p || which < 0 || which > p->nin) return nullptr;
    return &p->pat[which];
}

int femo_problem_pattern_info(const femo_problem *p, int which, int64_t info[4]) {
    const Pattern *P = get_pat(p, which);
    if (!P || !info) return set_err(FEMO_EINVAL, "femo_problem_pattern_info: bad selector");
    info[0] = P->nrows; info[1] = P->ncols; info[2] = P->nnz; info[3] = P->ncontrib;
    return FEMO_OK;
}
int femo_problem_pattern(const femo_problem *p, int which, int32_t *rowptr, int32_t *col) {
    const Pattern *P = get_pat(p, which);
    if (!P) return set_err(FEMO_EINVAL, "femo_problem_pattern: bad selector");
    if (rowptr) memcpy(rowptr, P->rowptr.data(), P->rowptr.size() * sizeof(int32_t));
    if (col) memcpy(col, P->col.data(), P->col.size() * sizeof(int32_t));
    return FEMO_OK;
}
int femo_problem_gather_map(const femo_problem *p, int which, int32_t *ptr, int32_t *src) {
    const Pattern *P = get_pat(p, which);
    if (!P) return set_err(FEMO_EINVAL, "femo_problem_gather_map: bad selector");
    if (ptr) memcpy(ptr, P->gptr.data(), P->gptr.size() * sizeof(int32_t));
    if (src) memcpy(src, P->gsrc.data(), P->gsrc.size() * sizeof(int32_t));
    return FEMO_OK;
}

static int set_bc_impl(femo_problem *p, const int32_t *dofs, const int32_t *list_ptr, int nlists, const double *g) {
    const int64_t N = p->state.ndofs;
    p->bc_mark.assign(N, 0);
    p->bc_diag.assign(N, 0.0);
    p->bc_g.assign(N, 0.0);
    for (int l = 0; l < nlists; ++l)
        for (int32_t k = list_ptr[l]; k < list_ptr[l + 1]; ++k) {
            int32_t d = dofs[k];
            if (d < 0 || d >= N) return set_err(FEMO_EINVAL, "femo_problem_set_bc: dof out of range");
            p->bc_mark[d] = 1;
            p->bc_diag[d] += 1.0;  // dolfinx set_diagonal adds once per dirichletbc object
        }
    if (g)
        for (int64_t i = 0; i < N; ++i)
            if (p->bc_mark[i]) p->bc_g[i] = g[i];
    const Pattern &P = p->pat[0];
    p->bcflag.assign(P.nnz, 0);
    std::vector<uint8_t> lift(N, 0);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < N; ++i) {
        bool any = p->bc_mark[i];
        for (int32_t t = P.rowptr[i]; t < P.rowptr[i + 1]; ++t) {
            int32_t j = P.col[t];
            if (p->bc_mark[i] || p->bc_mark[j]) p->bcflag[t] = (i == j) ? 2 : 1;
            any = any || p->bc_mark[j];
        }
        lift[i] = any;
    }
    p->lift_rows.clear();
    for (int64_t i = 0; i < N; ++i)
        if (lift[i]) p->lift_rows.push_back((int32_t)i);
    p->has_bc = nlists > 0 && !p->lift_rows.empty();
    if (p->uploaded) return push_bc(p);
    return FEMO_OK;
}

// coarse multigrid levels inherit Dirichlet rows geometrically: a coarse node is
// constrained when the fine node nearest to it is (homogeneous correction equation)
static int propagate_bc(femo_problem *root, int start) {
    const femo_problem *F = mg_level(root, start);
    for (size_t lv = (size_t)start; lv < root->mg.size(); ++lv) {
        femo_problem *C = root->mg[lv];
        if (C->replicated && F->slab.active) {
            // the first replicated level needs the marks of every rank: gathered on the device at the next set-up
            root->mg_bc_dirty = true;
            return FEMO_OK;
        }
        std::vector<int32_t> list;
        const int fnx = F->mesh.n[0], fny = F->mesh.n[1], cnx = C->mesh.n[0], cny = C->mesh.n[1];
        const int fnz = F->mesh.n[2], cnz = C->mesh.n[2];                          // 0 on planar lattices
        const bool zslab = cnz > 0;                                                 // slabs cut the last lattice axis
        const int fs0 = F->slab.active ? F->slab.crow0 : 0, cs0 = C->slab.active ? C->slab.crow0 : 0;
        const int fj0 = zslab ? 0 : fs0, cj0 = zslab ? 0 : cs0, fk0 = zslab ? fs0 : 0, ck0 = zslab ? cs0 : 0;
        const int fg = (!zslab && F->slab.active) ? F->slab.gny : fny, cg = (!zslab && C->slab.active) ? C->slab.gny : cny;
        const int fgz = (zslab && F->slab.active) ? F->slab.gny : fnz, cgz = (zslab && C->slab.active) ? C->slab.gny : cnz;
        for (int K = 0; K <= cnz; ++K)
        for (int J = 0; J <= cny; ++J)
            for (int I = 0; I <= cnx; ++I) {
                const int i = (int)std::llround((double)I * fnx / cnx);
                int j = (int)std::llround((double)(J + cj0) * fg / cg) - fj0;     // nearest fine row, local index
                j = std::min(std::max(j, 0), fny);                                 // ghost rows without a local parent: same column
                int k = cnz ? (int)std::llround((double)(K + ck0) * fgz / cgz) - fk0 : 0;
                k = std::min(std::max(k, 0), fnz);
                const int bs = F->state.block;
                for (int cc = 0; cc < bs; ++cc)
                    if (!F->bc_mark.empty() && F->bc_mark[(((int64_t)k * (fny + 1) + j) * (fnx + 1) + i) * bs + cc])
                        list.push_back((int32_t)((((int64_t)K * (cny + 1) + J) * (cnx + 1) + I) * bs + cc));
            }
        int32_t ptr[2] = {0, (int32_t)list.size()};
        int rc = set_bc_impl(C, list.data(), ptr, list.empty() ? 0 : 1, nullptr);
        if (rc) return rc;
        F = C;
    }
    return FEMO_OK;
}

int femo_problem_set_bc(femo_problem *p, const int32_t *dofs, const int32_t *list_ptr, int nlists, const double *g) {
    if (!p || nlists < 0 || (nlists > 0 && (!dofs || !list_ptr))) return set_err(FEMO_EINVAL, "femo_problem_set_bc: bad arguments");
    int rc = set_bc_impl(p, dofs, list_ptr, nlists, g);
    if (rc) return rc;
    return propagate_bc(p);
}

// ---- device residency -----------------------------------------------------
// What the static and work arenas hold is decided in one place: the layout walk lay_out_problem, which covers the fine
// level and then every coarse multigrid level (lay_out_level).  It runs twice (Arena, common.cuh): counting for
// femo_problem_device_bytes and placing for femo_problem_upload, so the size query and the layout cannot disagree.  The
// order of the reservations is the layout.  Host state derived while placing is set in place mode only, so the count
// pass writes nothing into the problem.
constexpr int kGmresRestart = 70;

// a matrix pattern (static): CSR, gather map, transpose permutation, SpMV row blocks, and the transposed CSR of a
// rectangular pattern; a square pattern shares rowptr / col / row blocks with its transpose
static void lay_out_pattern(Arena &st, const Pattern &P, DevPattern &D) {
    put(st, D.rowptr, P.rowptr);
    put(st, D.col, P.col);
    put(st, D.gptr, P.gptr);
    put(st, D.gsrc, P.gsrc);
    put(st, D.t_perm, P.t_perm);
    if (!P.square_symmetric) {
        put(st, D.t_rowptr, P.t_rowptr);
        put(st, D.t_col, P.t_col);
    }
    put(st, D.rb, P.rb);
    if (!P.square_symmetric) put(st, D.t_rb, P.t_rb);
    if (st.counting()) return;
    D.nrb = (int)P.rb.size() - 1;
    if (P.square_symmetric) {
        D.t_rowptr = D.rowptr;
        D.t_col = D.col;
        D.t_rb = D.rb;
        D.t_nrb = D.nrb;
    } else {
        D.t_nrb = (int)P.t_rb.size() - 1;
    }
}

// Dirichlet arrays (static): per-nnz flag, marker, value, multiplicity, lifted rows.  Reserved with or without
// conditions: femo_problem_set_bc may come after upload, and push_bc fills them.
static void lay_out_bc(Arena &st, femo_problem *c) {
    const int64_t N = c->state.ndofs;
    st.take(c->dpat[0].bcflag, c->pat[0].nnz);
    st.take(c->d_bc_mark, N);
    st.take(c->d_bc_g, N);
    st.take(c->d_bc_diag, N);
    st.take(c->d_lift_rows, N);
}

// a coarse multigrid level in the root's arenas: mesh, Jacobian pattern and Dirichlet arrays (static); matrix values,
// smoother and V-cycle vectors, and on the coarsest level the explicit inverse (work)
static void lay_out_level(femo_problem *c, bool coarsest, Arena &st, Arena &wk) {
    const Mesh &M = c->mesh;
    const int64_t N = c->state.ndofs;
    put(st, c->d_coords, M.coords);
    put_soa(st, c->d_cellsT, M.cells, M.nvpc);
    put(st, c->d_fb_cell, c->fb_cell);
    put(st, c->d_fb_local, c->fb_local);
    lay_out_pattern(st, c->pat[0], c->dpat[0]);
    lay_out_bc(st, c);
    femo_mg_level &L = c->mgl;
    wk.take(L.vals, c->pat[0].nnz);
    wk.take(L.vals32, fp32_copy_len(c));
    lay_out_matfree(c, st, wk);
    for (double **v : {&L.dinv, &L.x, &L.b, &L.r, &L.d, &L.q, &L.u}) wk.take(*v, N);
    wk.take(L.m, std::max<int64_t>(1, M.ncells));
    wk.take(L.fb, N);
    wk.take(L.fx, N);
    wk.take(c->d_partials, 3 * kMaxPartials);
    wk.take(c->d_scalars, S_COUNT);
    if (coarsest) {
        wk.take(L.dense, (size_t)N * N);
        wk.take(L.dense_tmp, (size_t)N * N);
    }
}

static void lay_out_problem(femo_problem *p, Arena &st, Arena &wk) {
    const Mesh &M = p->mesh;
    const int64_t N = p->state.ndofs;
    put(st, p->d_coords, M.coords);
    put_soa(st, p->d_cellsT, M.cells, M.nvpc);
    put(st, p->d_fb_cell, p->fb_cell);
    put(st, p->d_fb_local, p->fb_local);
    put(st, p->d_cell_tag, M.cell_tag);
    if ((p->family == FEMO_FAMILY_NLPOISSON_P1 || p->family == FEMO_FAMILY_NLPOISSON_P2) && M.kind == MESH_TRI && M.lattice &&
        !p->jac_only && !getenv("FEMO_NO_UEX_TABLE")) {
        // u_ex = sin(2 pi x) sin(pi y) at x0 + dx_q: cos / sin of the offsets of the 49 points in both triangle types
        const double hx = (M.hi[0] - M.lo[0]) / (double)M.n[0];
        const double hy = (M.hi[1] - M.lo[1]) / (double)(p->slab.active ? p->slab.gny : M.n[1]);
        const double pi = 3.141592653589793;
        std::vector<double> gx, gw, tab(2 * 49 * 4);
        gauss_legendre_01(7, gx, gw);
        for (int t = 0; t < 2; ++t)
            for (int i = 0; i < 7; ++i)
                for (int j = 0; j < 7; ++j) {
                    const double xi = gx[i], et = gx[j] * (1.0 - gx[i]);          // same points as c_tri49
                    const double dx = t == 0 ? hx * (xi + et) : hx * et;          // lower: e1 = (hx,0); upper: e1 = (0,hy); e2 = (hx,hy)
                    const double dy = t == 0 ? hy * et : hy * (xi + et);
                    double *o = &tab[((size_t)t * 49 + 7 * i + j) * 4];
                    o[0] = std::cos(2.0 * pi * dx); o[1] = std::sin(2.0 * pi * dx);
                    o[2] = std::cos(pi * dy); o[3] = std::sin(pi * dy);
                }
        put(st, p->d_uex_tab, tab);
        if (!st.counting()) p->h_uex_tab = std::move(tab);   // the moved buffer stays alive for the pending copy
    }
    if (p->state.element == EL_RMP || p->state.element == EL_P2) put_soa(st, p->d_edgesT, M.cell_edges, 3);
    if (p->state.element == EL_P2) {
        put(st, p->d_edge_verts, M.edge_verts);
        put(st, p->d_vptr, p->vptr);
        put(st, p->d_vedge, p->vedge);
    }
    for (int w = 0; w <= p->nin; ++w) lay_out_pattern(st, p->pat[w], p->dpat[w]);
    if (!p->pat[0].b_perm.empty()) {
        const Pattern &P = p->pat[0];
        DevPattern &D = p->dpat[0];
        put(st, D.b_rowptr, P.b_rowptr);
        put(st, D.b_col, P.b_col);
        put(st, D.b_perm, P.b_perm);
        put(st, D.b_rb, P.b_rb);
        if (!st.counting()) D.nbrb = (int)P.b_rb.size() - 1;
    }
    for (int m = 1; m < 4; ++m) {
        if (p->vm_state[m].ptr.empty()) continue;
        put(st, p->dvm_state[m].ptr, p->vm_state[m].ptr);
        put(st, p->dvm_state[m].src, p->vm_state[m].src);
    }
    for (int i = 0; i < p->nin; ++i) {
        put(st, p->dvm_in[i].ptr, p->vm_in[i].ptr);
        put(st, p->dvm_in[i].src, p->vm_in[i].src);
    }
    lay_out_bc(st, p);

    size_t scratch = 0, tv = 0;
    for (int w = 0; w <= p->nin; ++w) {
        scratch = std::max<size_t>(scratch, p->pat[w].scratch_len);
        tv = std::max<size_t>(tv, p->pat[w].nnz);
    }
    for (int m = 1; m < 4; ++m) scratch = std::max<size_t>(scratch, p->vm_state[m].scratch_len);
    for (int i = 0; i < p->nin; ++i) scratch = std::max<size_t>(scratch, p->vm_in[i].scratch_len);
    scratch = std::max<size_t>(scratch, (size_t)M.ncells);
    const int64_t nnz = p->pat[0].nnz;
    wk.take(p->d_scratch, scratch);
    wk.take(p->d_partials, 3 * kMaxPartials);
    wk.take(p->d_scalars, S_COUNT);
    for (double **v : {&p->kr_r, &p->kr_p, &p->kr_q, &p->kr_dinv, &p->kr_z, &p->kr_w, &p->nt_b, &p->nt_dx}) wk.take(*v, N);
    wk.take(p->nt_vals, nnz);
    wk.take(p->nt_vals_bc, nnz);
    wk.take(p->d_tvals, tv);
    if (!p->pat[0].b_perm.empty()) wk.take(p->d_bvals, nnz);
    wk.take(p->kr_d, N);
    if (!p->mg.empty()) {
        wk.take(p->mgl.vals32, fp32_copy_len(p));
        wk.take(p->d_mgops, kMgFusedMaxOps);
        DiaMat A;   // fp64 planes of the fine-level operator for the Krylov recurrence (lattice stencil problems)
        if (dia_offsets(p, A)) wk.take(p->mgl.dia64, (size_t)A.nd * (size_t)A.np);
    }
    lay_out_matfree(p, st, wk);
    if (!p->symmetric) {   // GMRES: Krylov basis, a spare vector, multi-dot partials
        wk.take(p->gm_basis, (size_t)(kGmresRestart + 1) * N);
        wk.take(p->wk_extra, N);
        wk.take(p->d_partials_big, (size_t)(kGmresRestart + 1) * kMaxPartials);
    }
    if (N <= kMgDenseMax) {   // explicit inverse (precond 3)
        wk.take(p->d_dense, (size_t)N * N);
        wk.take(p->d_dense_tmp, (size_t)N * N);
    }
    for (size_t l = 0; l < p->mg.size(); ++l) lay_out_level(p->mg[l], l + 1 == p->mg.size(), st, wk);
    if (wk.counting()) return;
    p->scratch_len = scratch;
    p->tvals_len = tv;
    if (!p->symmetric) p->gm_restart = kGmresRestart;
}

// both figures are exact: the count pass of the walk that femo_problem_upload places
int femo_problem_device_bytes(const femo_problem *p, size_t *static_bytes, size_t *work_bytes) {
    if (!p || !static_bytes || !work_bytes) return set_err(FEMO_EINVAL, "femo_problem_device_bytes: null");
    refresh_env();
    Arena st, wk;   // no buffers: the walk only counts, so *p stays as it is
    lay_out_problem(const_cast<femo_problem *>(p), st, wk);
    *static_bytes = st.used;
    *work_bytes = wk.used;
    return FEMO_OK;
}

int femo_problem_upload(femo_problem *p, int device, void *stream, void *d_static, size_t static_bytes, void *d_work,
                        size_t work_bytes) {
    if (!p || !d_static || !d_work) return set_err(FEMO_EINVAL, "femo_problem_upload: null");
    if (femo_device_count() <= device || device < 0)
        return set_err(FEMO_ENODEVICE, "femo_problem_upload: no such CUDA device; this engine has no CPU path");
    size_t sb, wb;
    femo_problem_device_bytes(p, &sb, &wb);
    if (static_bytes < sb || work_bytes < wb) return set_err(FEMO_EINVAL, "femo_problem_upload: arenas smaller than femo_problem_device_bytes");
    FEMO_CUDA(cudaSetDevice(device));
    p->device = device;
    p->stream = (cudaStream_t)stream;
    cudaDeviceProp prop;
    FEMO_CUDA(cudaGetDeviceProperties(&prop, device));
    p->num_sms = prop.multiProcessorCount;
    if (!p->stream2) {
        int lo_prio = 0, hi_prio = 0;
        FEMO_CUDA(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
        FEMO_CUDA(cudaStreamCreateWithPriority(&p->stream2, cudaStreamNonBlocking, hi_prio));
        FEMO_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
        FEMO_CUDA(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
    }
    Arena st(d_static, static_bytes, p->stream), wk(d_work, work_bytes, p->stream);
    lay_out_problem(p, st, wk);
    int rc;
    if ((rc = st.check(sb, "femo_problem_upload: static arena")) || (rc = wk.check(wb, "femo_problem_upload: work arena"))) return rc;
    if ((rc = push_bc(p))) return rc;

    // quadrature tables
    {
        double tri6[6][3];
        const double s10 = std::sqrt(10.0), tt = std::sqrt(38.0 - 44.0 * std::sqrt(2.0 / 5.0));
        const double a[2] = {(8.0 - s10 + tt) / 18.0, (8.0 - s10 - tt) / 18.0};
        const double sw = std::sqrt(213125.0 - 53320.0 * s10);
        const double wgt[2] = {(620.0 + sw) / 3720.0, (620.0 - sw) / 3720.0};
        for (int k = 0; k < 2; ++k) {
            const double b = 1.0 - 2.0 * a[k];
            const double pts[3][2] = {{a[k], a[k]}, {a[k], b}, {b, a[k]}};
            for (int j = 0; j < 3; ++j) {
                tri6[3 * k + j][0] = pts[j][0];
                tri6[3 * k + j][1] = pts[j][1];
                tri6[3 * k + j][2] = 0.5 * wgt[k];
            }
        }
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_tri6, tri6, sizeof(tri6), 0, cudaMemcpyHostToDevice, p->stream));
        const double tri3[3][3] = {{1.0 / 6.0, 1.0 / 6.0, 1.0 / 6.0}, {1.0 / 6.0, 2.0 / 3.0, 1.0 / 6.0}, {2.0 / 3.0, 1.0 / 6.0, 1.0 / 6.0}};
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_tri3, tri3, sizeof(tri3), 0, cudaMemcpyHostToDevice, p->stream));
        std::vector<double> x, w;
        gauss_legendre_01(5, x, w);
        double gl5[5][2];
        for (int i = 0; i < 5; ++i) { gl5[i][0] = x[i]; gl5[i][1] = w[i]; }
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_gl5, gl5, sizeof(gl5), 0, cudaMemcpyHostToDevice, p->stream));
        gauss_legendre_01(7, x, w);
        double t49[49][3];
        for (int i = 0; i < 7; ++i)
            for (int j = 0; j < 7; ++j) {
                t49[7 * i + j][0] = x[i];
                t49[7 * i + j][1] = x[j] * (1.0 - x[i]);
                t49[7 * i + j][2] = w[i] * w[j] * (1.0 - x[i]);
            }
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_tri49, t49, sizeof(t49), 0, cudaMemcpyHostToDevice, p->stream));
        std::vector<double> x5, w5, x6, w6;
        gauss_legendre_01(5, x5, w5);
        double t25[25][3];
        for (int i = 0; i < 5; ++i)
            for (int j = 0; j < 5; ++j) {
                t25[5 * i + j][0] = x5[i];
                t25[5 * i + j][1] = x5[j] * (1.0 - x5[i]);
                t25[5 * i + j][2] = w5[i] * w5[j] * (1.0 - x5[i]);
            }
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_tri25, t25, sizeof(t25), 0, cudaMemcpyHostToDevice, p->stream));
        gauss_legendre_01(6, x6, w6);
        double gl6[6][2];
        for (int i = 0; i < 6; ++i) { gl6[i][0] = x6[i]; gl6[i][1] = w6[i]; }
        FEMO_CUDA(cudaMemcpyToSymbolAsync(c_gl6, gl6, sizeof(gl6), 0, cudaMemcpyHostToDevice, p->stream));
        FEMO_CUDA(cudaStreamSynchronize(p->stream));
    }

    for (femo_problem *c : p->mg) {   // coarse levels run on the fine level's streams and reuse its element scratch
        c->device = p->device;
        c->stream = p->stream;
        c->stream2 = p->stream2;
        c->ev_fork = p->ev_fork;
        c->ev_join = p->ev_join;
        c->num_sms = p->num_sms;
        c->d_scratch = p->d_scratch;
        c->scratch_len = p->scratch_len;
        FEMO_CUDA(cudaMemsetAsync(c->d_scalars, 0, sizeof(double) * S_COUNT, p->stream));
        if (!c->h_pinned) FEMO_CUDA(cudaMallocHost((void **)&c->h_pinned, sizeof(double) * 128));
        if ((rc = push_bc(c))) return rc;
        c->uploaded = true;
    }
    FEMO_CUDA(cudaMemsetAsync(p->d_scalars, 0, sizeof(double) * S_COUNT, p->stream));
    if (!p->h_pinned) FEMO_CUDA(cudaMallocHost((void **)&p->h_pinned, sizeof(double) * 128));
    FEMO_CUDA(cudaStreamSynchronize(p->stream));
    p->uploaded = true;
    return FEMO_OK;
}

int femo_set_coefficient(femo_problem *p, int slot, const double *d_values, int64_t n) {
    if (!p || slot < 0 || slot > p->nin + p->naux) return set_err(FEMO_EINVAL, "femo_set_coefficient: bad slot");
    int64_t want = (slot == 0) ? p->state.ndofs : (slot <= p->nin ? p->in[slot - 1].ndofs : p->aux[slot - 1 - p->nin].ndofs);
    if (n != want) return set_err(FEMO_EINVAL, "femo_set_coefficient: size does not match the slot's space");
    p->coef[slot] = d_values;
    p->coefn[slot] = n;
    return FEMO_OK;
}

int femo_problem_launch_count(const femo_problem *p, long long *count) {
    if (!p || !count) return set_err(FEMO_EINVAL, "femo_problem_launch_count: null");
    *count = total_launches(p);
    return FEMO_OK;
}

int femo_problem_graph_replays(const femo_problem *p, long long *count) {
    if (!p || !count) return set_err(FEMO_EINVAL, "femo_problem_graph_replays: null");
    *count = p->graph_replays;
    return FEMO_OK;
}

// ---- multi-GPU communicator ------------------------------------------------
int femo_comm_unique_id(char id[128]) {
    int rc = nccl_load();
    if (rc) return rc;
    ncclUniqueId u;
    FEMO_NCCL(g_comm.api.GetUniqueId(&u));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    memcpy(id, &u, 128);
    return FEMO_OK;
}

int femo_comm_init(const char id[128], int rank, int nranks, int device) {
    if (!id || nranks < 1 || rank < 0 || rank >= nranks) return set_err(FEMO_EINVAL, "femo_comm_init: bad arguments");
    if (g_comm.active) return set_err(FEMO_ESTATE, "femo_comm_init: communicator already initialised");
    if (femo_device_count() <= device || device < 0) return set_err(FEMO_ENODEVICE, "femo_comm_init: no such CUDA device");
    int rc = nccl_load();
    if (rc) return rc;
    FEMO_CUDA(cudaSetDevice(device));
    ncclUniqueId u;
    memcpy(&u, id, 128);
    FEMO_NCCL(g_comm.api.CommInitRank(&g_comm.comm, nranks, u, rank));
    g_comm.rank = rank;
    g_comm.nranks = nranks;
    g_comm.active = nranks > 1;
    return FEMO_OK;
}

/* peer-memory transport (link.cuh): every rank creates its window and publishes the 64-byte IPC handle ... */
int femo_link_create(int device, size_t halo_cap, size_t gather_cap, char handle[64]) {
    if (!handle) return set_err(FEMO_EINVAL, "femo_link_create: null handle");
    if (femo_device_count() <= device || device < 0) return set_err(FEMO_ENODEVICE, "femo_link_create: no such CUDA device");
    if (g_link.local) return set_err(FEMO_ESTATE, "femo_link_create: window already created");
    FEMO_CUDA(cudaSetDevice(device));
    g_link.lay.halo_cap = halo_cap ? halo_cap : ((size_t)1 << 18);       // 16-byte lines: 4 slots x 4 MB
    g_link.lay.gather_cap = gather_cap ? gather_cap : ((size_t)1 << 21);   // 2 buffers x 32 MB
    const size_t bytes = g_link.lay.bytes();
    FEMO_CUDA(cudaMalloc((void **)&g_link.local, bytes));
    FEMO_CUDA(cudaMemset(g_link.local, 0, bytes));
    FEMO_CUDA(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    FEMO_CUDA(cudaIpcGetMemHandle(&h, g_link.local));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
    memcpy(handle, &h, 64);
    g_link.device = device;
    return FEMO_OK;
}

/* ... and maps the windows of all ranks (handles = nranks x 64 bytes, rank-major; the own entry is not opened). */
int femo_link_open(const char *handles, int rank, int nranks) {
    if (!handles || nranks < 1 || nranks > kLinkMaxRanks || rank < 0 || rank >= nranks)
        return set_err(FEMO_EINVAL, "femo_link_open: bad arguments (at most 16 ranks)");
    if (!g_link.local) return set_err(FEMO_ESTATE, "femo_link_open: call femo_link_create first");
    if (g_comm.active) return set_err(FEMO_ESTATE, "femo_link_open: a communicator is already active");
    FEMO_CUDA(cudaSetDevice(g_link.device));
    for (int r = 0; r < nranks; ++r) {
        if (r == rank) {
            g_link.win[r] = g_link.local;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + 64 * (size_t)r, 64);
        void *ptr = nullptr;
        FEMO_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        g_link.win[r] = (char *)ptr;
    }
    g_link.rank = rank;
    g_link.nranks = nranks;
    g_link.seq_halo = g_link.seq_ar = g_link.seq_gather = 0;
    g_link.active = nranks > 1;
    g_comm.rank = rank;
    g_comm.nranks = nranks;
    g_comm.active = nranks > 1;
    return FEMO_OK;
}

/* 1 when a spin of the transport timed out since the window was created (the results after that are invalid) */
int femo_link_error(void) {
    if (!g_link.local) return 0;
    int e = 0;
    if (cudaMemcpy(&e, g_link.local + LinkLayout::kErr, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    return e;
}

int femo_comm_finalize(void) {
    if (g_link.local) {
        cudaSetDevice(g_link.device);
        cudaDeviceSynchronize();
        for (int r = 0; r < g_link.nranks; ++r)
            if (r != g_link.rank && g_link.win[r]) cudaIpcCloseMemHandle(g_link.win[r]);
        cudaFree(g_link.local);
        g_link = Link();
    }
    if (g_comm.comm) {
        g_comm.api.CommDestroy(g_comm.comm);
        g_comm.comm = nullptr;
    }
    g_comm.active = false;
    return FEMO_OK;
}

int femo_comm_stats(long long stats[2]) {
    if (!stats) return set_err(FEMO_EINVAL, "femo_comm_stats: null");
    stats[0] = g_comm.halo_exchanges;
    stats[1] = g_comm.allreduces;
    return FEMO_OK;
}

/* Unstructured partitions (femo_b200/partition.py): see include/femo_b200.h. */
int femo_problem_set_partition(femo_problem *p, int64_t n_owned_nodes, int64_t n_owned_cells, int64_t blk_nodes, int64_t n_send,
                               const int32_t *send_nodes, int64_t n_ghost, const int32_t *ghost_src_nodes, void *d_buf,
                               int64_t *bytes) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!bytes || n_owned_nodes < 0 || n_owned_cells < 0 || blk_nodes < 0 || (n_send && !send_nodes) || (n_ghost && !ghost_src_nodes))
        return set_err(FEMO_EINVAL, "femo_problem_set_partition: bad arguments");
    if (p->slab.active) return set_err(FEMO_ESTATE, "femo_problem_set_partition: slab problems carry their own partition");
    const int b = p->state.block;
    const int64_t N = p->state.ndofs, nn = N / b;
    if (n_owned_nodes + n_ghost != nn || n_owned_cells > p->mesh.ncells)
        return set_err(FEMO_EINVAL, "femo_problem_set_partition: owned + ghost nodes must cover the local mesh (owned first)");
    const int R = std::max(1, g_comm.nranks);
    const int64_t ns = n_send * b, ng = n_ghost * b, blk = std::max<int64_t>(1, blk_nodes * b);
    GenPart &G = p->gpart;
    auto lay_out = [&](Arena &A) {   // the buffer's layout walk: send indices, ghost sources, the gathered buffer of all ranks
        A.take(G.d_send_idx, std::max<int64_t>(ns, 1));
        A.take(G.d_ghost_src, std::max<int64_t>(ng, 1));
        A.take(G.d_gather, (size_t)blk * R);
    };
    Arena count;
    lay_out(count);
    if (!d_buf) {
        *bytes = (int64_t)count.used;
        return FEMO_OK;
    }
    if (*bytes < (int64_t)count.used) return set_err(FEMO_EINVAL, "femo_problem_set_partition: buffer smaller than the size query reported");
    G.send_idx.resize(ns);
    G.ghost_src.resize(ng);
    for (int64_t k = 0; k < n_send; ++k) {
        if (send_nodes[k] < 0 || send_nodes[k] >= n_owned_nodes) return set_err(FEMO_EINVAL, "femo_problem_set_partition: send list entry is not an owned node");
        for (int c = 0; c < b; ++c) G.send_idx[k * b + c] = send_nodes[k] * b + c;
    }
    for (int64_t k = 0; k < n_ghost; ++k) {
        const int64_t q = blk_nodes ? ghost_src_nodes[k] / blk_nodes : 0, pos = blk_nodes ? ghost_src_nodes[k] % blk_nodes : 0;
        if (q < 0 || q >= R) return set_err(FEMO_EINVAL, "femo_problem_set_partition: ghost source outside the gathered buffer");
        for (int c = 0; c < b; ++c) G.ghost_src[k * b + c] = (int32_t)(q * blk + pos * b + c);
    }
    G.n_owned_dofs = n_owned_nodes * b;
    G.n_owned_cells = n_owned_cells;
    G.blk = blk;
    Arena A(d_buf, (size_t)*bytes);
    lay_out(A);
    FEMO_CUDA(cudaSetDevice(p->device));
    if (ns) FEMO_CUDA(cudaMemcpy(G.d_send_idx, G.send_idx.data(), ns * 4, cudaMemcpyHostToDevice));
    if (ng) FEMO_CUDA(cudaMemcpy(G.d_ghost_src, G.ghost_src.data(), ng * 4, cudaMemcpyHostToDevice));
    FEMO_CUDA(cudaMemset(G.d_gather, 0, (size_t)blk * R * 8));
    p->own_off = 0;
    p->own_n = G.n_owned_dofs;
    p->cown_off = 0;
    p->cown_n = n_owned_cells;
    G.active = true;
    return FEMO_OK;
}

/* refresh the ghost rows of a state-space (kind 0) or cell-wise input (kind 1) vector */
int femo_halo_exchange(femo_problem *p, double *d_v, int kind) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_v) return set_err(FEMO_EINVAL, "femo_halo_exchange: null");
    return kind == 0 ? halo_nodes(p, d_v) : halo_cells(p, d_v);
}

// arguments of the node-centric lattice kernels (lattice_asm.cuh)
static void lattice_args(femo_problem *p, LatJacArgs &A, LatGeom &G) {
    const DevPattern &D = p->dpat[0];
    A.T = tri_args(p, nullptr);
    A.nx = p->mesh.n[0]; A.ny = p->mesh.n[1];
    A.ext_bottom = !p->slab.active || p->slab.rank == 0;
    A.ext_top = !p->slab.active || p->slab.rank == p->slab.nranks - 1;
    A.rowptr = D.rowptr; A.col = D.col; A.bcflag = D.bcflag; A.bc_diag = p->d_bc_diag;
    A.out = A.out_bc = nullptr;
    // P1 gradients of the two congruent triangle types of the uniform lattice
    const double hx = (p->mesh.hi[0] - p->mesh.lo[0]) / (double)p->mesh.n[0];
    const double hy = (p->mesh.hi[1] - p->mesh.lo[1]) / (double)(p->slab.active ? p->slab.gny : p->mesh.n[1]);
    const double gl[3][2] = {{-1.0 / hx, 0.0}, {1.0 / hx, -1.0 / hy}, {0.0, 1.0 / hy}};
    const double gu[3][2] = {{0.0, -1.0 / hy}, {-1.0 / hx, 1.0 / hy}, {1.0 / hx, 0.0}};
    memcpy(G.gl, gl, sizeof(gl));
    memcpy(G.gu, gu, sizeof(gu));
    G.a2 = hx * hy;
}

// Node-centric Jacobian of a lattice level.  with_dia: also write the level operator straight into the DIA planes of
// the multigrid solve (fp32 + scaling plane, dinv, Gershgorin maxima -> S_TMP2; fp64 planes on level 0), BC'd copy when
// dia_bc.  d_vals / d_vals_bc may both be null then (the CSR values are not needed by a DIA-only level).
static int lattice_jacobian(femo_problem *p, double *d_vals, double *d_vals_bc, bool with_dia, bool dia_bc) {
    int rc;
    if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
    LatJacArgs A;
    LatGeom G;
    lattice_args(p, A, G);
    A.out = d_vals; A.out_bc = d_vals_bc;
    LatDiaOut O;
    femo_mg_level &M = p->mgl;
    const int g = grid_for(p->state.ndofs);
    if (with_dia) {
        DiaMat D;
        if (!dia_offsets(p, D) || !M.vals32 || !M.dinv) return set_err(FEMO_ESTATE, "lattice_jacobian: level has no DIA storage");
        if ((size_t)g > p->scratch_len) return set_err(FEMO_ESTATE, "lattice_jacobian: scratch too small for the partial maxima");
        D.v = M.vals32;
        O.planes32 = M.vals32; O.planes64 = M.dia64; O.dinv = M.dinv; O.gpart = p->d_scratch;
        O.np = D.np; O.o0 = p->own_off; O.o1 = p->own_off + p->own_n; O.use_bc = dia_bc ? 1 : 0;
        M.dia = D;
    }
    // interior nodes (lean instantiation) + the two outer rings with the Nitsche facet rows (lattice_asm.cuh)
    const int gp = grid_for(lattice_band_count(A.nx, A.ny));
    if (with_dia && (size_t)(g + gp) > p->scratch_len) return set_err(FEMO_ESTATE, "lattice_jacobian: scratch too small for the partial maxima");
    k_nlpoisson_p1_node_jac<false><<<g, kThreads, 0, p->stream>>>(A, G, O);
    O.gpart_off = g;
    k_nlpoisson_p1_node_jac<true><<<gp, kThreads, 0, p->stream>>>(A, G, O);
    p->launches += 2;
    FEMO_CHECK_LAUNCH();
    if (with_dia) {
        k_max_finalize<<<1, kThreads, 0, p->stream>>>(p->d_scratch, g + gp, p->d_scalars, S_TMP2);
        p->launches++;
        FEMO_CHECK_LAUNCH();
        M.dia_valid = true;
        M.dia64_valid = M.dia64 != nullptr;
        return halo_nodes_f32(p, M.vals32 + (size_t)M.dia.nd * M.dia.np);
    }
    return FEMO_OK;
}

// ---- assembly -------------------------------------------------------------
int femo_assemble_residual(femo_problem *p, double *d_out) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_out) return set_err(FEMO_EINVAL, "femo_assemble_residual: null output");
    if (p->lattice_fast && p->res_mask == 3 && !g_env.no_lattice_asm) {
        if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
        if ((rc = need_coef(p, 1, p->in[0].ndofs, "input 0"))) return rc;
        LatJacArgs A;
        LatGeom G;
        lattice_args(p, A, G);
        k_nlpoisson_p1_node_res<false><<<grid_for(p->state.ndofs), kThreads, 0, p->stream>>>(A, G, d_out);
        k_nlpoisson_p1_node_res<true><<<grid_for(lattice_band_count(A.nx, A.ny)), kThreads, 0, p->stream>>>(A, G, d_out);
        p->launches += 2;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    if ((rc = run_elements(p, OP_RES, p->res_mask))) return rc;
    return segreduce(p, p->dvm_state[p->res_mask], p->state.ndofs, d_out);
}

int femo_assemble_jacobian(femo_problem *p, double *d_vals, double *d_vals_bc) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_vals && !d_vals_bc) return set_err(FEMO_EINVAL, "femo_assemble_jacobian: both outputs null");
    const DevPattern &D = p->dpat[0];
    const int64_t nnz = p->pat[0].nnz;
    if (p->mgl.k0 && p->mgl.ec && p->family == FEMO_FAMILY_SIMP_HEX8 && p->jac_mask == 1) {   // uniform lattice fast path
        if ((rc = need_coef(p, 1, p->in[0].ndofs, "input 0"))) return rc;
        const int64_t nc = p->mesh.ncells;
        k_pow_cells<<<grid_for(nc), kThreads, 0, p->stream>>>(p->coef[1], p->params[4], p->mgl.ec, nc);
        k_segreduce_jac_k0<<<grid_for(nnz), kThreads, 0, p->stream>>>(D.gptr, D.gsrc, p->mgl.k0, p->mgl.ec, (uint32_t)nc, D.bcflag,
                                                                      D.col, p->d_bc_diag, d_vals, d_vals_bc, nnz);
        p->launches += 2;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    if (p->lattice_fast && !g_env.no_lattice_asm) {   // right-diagonal lattice: node-centric rows, no scratch round trip
        if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
        return lattice_jacobian(p, d_vals, d_vals_bc, false, false);
    }
    if ((rc = run_elements(p, OP_JAC, p->jac_mask))) return rc;
    k_segreduce_jac<<<grid_for(nnz), kThreads, 0, p->stream>>>(D.gptr, D.gsrc, p->d_scratch,
                                                               D.bcflag, D.col, p->d_bc_diag,
                                                               d_vals, d_vals_bc, nnz);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

int femo_assemble_dRdm(femo_problem *p, int slot, double *d_vals) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (slot < 0 || slot >= p->nin || !d_vals) return set_err(FEMO_EINVAL, "femo_assemble_dRdm: bad slot/output");
    if ((rc = run_elements(p, OP_DRDM, p->drdm_mask, slot))) return rc;     // multi-input families read the slot
    const DevPattern &D = p->dpat[1 + slot];
    const int64_t nnz = p->pat[1 + slot].nnz;
    k_segreduce<<<grid_for(nnz), kThreads, 0, p->stream>>>(D.gptr, D.gsrc, p->d_scratch, d_vals, nnz);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

static int lifted_rhs(femo_problem *p, const double *d_vals, double *d_b, const double *x0, double scale) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_b) return set_err(FEMO_EINVAL, "lifted rhs: null output");
    if ((rc = femo_assemble_residual(p, d_b))) return rc;
    if (p->has_bc) {
        if (!d_vals) return set_err(FEMO_EINVAL, "lifted rhs: Jacobian values required for lifting");
        const int64_t nl = (int64_t)p->lift_rows.size();
        const DevPattern &D = p->dpat[0];
        k_newton_rhs<<<grid_for(nl), kThreads, 0, p->stream>>>(p->d_lift_rows, nl, D.rowptr, D.col, d_vals, p->d_bc_mark,
                                                               p->d_bc_g, x0, d_b, scale);
        p->launches++;
        FEMO_CHECK_LAUNCH();
    }
    return FEMO_OK;
}

int femo_newton_rhs(femo_problem *p, const double *d_vals, double *d_b) {
    if (!p) return set_err(FEMO_EINVAL, "null problem");
    return lifted_rhs(p, d_vals, d_b, p->coef[0], -1.0);
}

int femo_assemble_system_rhs(femo_problem *p, const double *d_vals, double *d_b) {
    return lifted_rhs(p, d_vals, d_b, nullptr, 1.0);
}

int femo_assemble_output(femo_problem *p, int out_id, double *h_value) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (out_id < 0 || out_id >= p->nout || !h_value) return set_err(FEMO_EINVAL, "femo_assemble_output: bad output id");
    const int om = p->out_mask[out_id];
    if ((rc = run_elements(p, OP_OUT, om, out_id))) return rc;
    const int64_t n = ((om & 1) ? p->mesh.ncells : 0) + ((om & 2) ? (int64_t)p->fb_cell.size() : 0);
    // on several GPUs every cell is summed by the rank that owns it
    const double *src = p->d_scratch;
    int64_t cnt = n;
    if (partitioned(p)) {
        if (om == 1) {
            src += p->cown_off;
            cnt = p->cown_n;
        } else if (p->gpart.active) {
            return set_err(FEMO_EINVAL, "facet functionals are not partitioned on unstructured meshes");
        } else if (om == 2) {           // facets are sorted by cell: the owned ones are a suffix
            src += p->fown_off;
            cnt = (int64_t)p->fb_cell.size() - p->fown_off;
        } else {
            return set_err(FEMO_EINVAL, "mixed cell + facet functionals are not partitioned");
        }
    }
    int g = red_grid(p, cnt);
    k_sum<<<g, kThreads, 0, p->stream>>>(src, cnt, p->d_partials);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    if ((rc = reduce_to(p, p->d_partials, nullptr, g, S_TMP1, 0))) return rc;
    return read_scalars(p, S_TMP1, 1, h_value);
}

int femo_assemble_output_grad(femo_problem *p, int out_id, int slot, double *d_out) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (out_id < 0 || out_id >= p->nout || !d_out || slot < 0 || slot > p->nin)
        return set_err(FEMO_EINVAL, "femo_assemble_output_grad: bad arguments");
    int mask = (slot == 0) ? p->out_du_mask[out_id] : p->out_dm_mask[out_id];
    if (p->family == FEMO_FAMILY_RM_PLATE && slot == 2) mask = 0;          // no output depends on the load
    const int64_t n = (slot == 0) ? p->state.ndofs : p->in[slot - 1].ndofs;
    if (mask == 0) {   // the functional does not depend on this argument
        FEMO_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * n, p->stream));
        return FEMO_OK;
    }
    if (slot == 0) {
        if ((rc = run_elements(p, OP_OUT_DU, mask, out_id))) return rc;
        return segreduce(p, p->dvm_state[mask], n, d_out);
    }
    if ((rc = run_elements(p, OP_OUT_DM, mask, out_id))) return rc;
    return segreduce(p, p->dvm_in[slot - 1], n, d_out);
}

/* OutputOperation.compute + compute_derivatives wrt the state (output_model.py:69-87) in ONE quadrature pass:
 * functional value and dJ/du share every evaluation point, so the fused pass halves the most expensive element
 * kernel of the nonlinear Poisson family (49-point rule, analytic u_ex).  Other families run the two passes. */
int femo_assemble_output_and_grad(femo_problem *p, int out_id, double *h_value, double *d_dJdu) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (out_id < 0 || out_id >= p->nout || !h_value || !d_dJdu) return set_err(FEMO_EINVAL, "femo_assemble_output_and_grad: bad arguments");
    if (p->family != FEMO_FAMILY_NLPOISSON_P1 || p->out_mask[out_id] != 1 || p->out_du_mask[out_id] != 1) {
        if ((rc = femo_assemble_output(p, out_id, h_value))) return rc;
        return femo_assemble_output_grad(p, out_id, 0, d_dJdu);
    }
    if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
    if ((rc = need_coef(p, 1, p->in[0].ndofs, "input 0"))) return rc;
    const int64_t nc = p->mesh.ncells;
    if ((size_t)(4 * nc) > p->scratch_len) return set_err(FEMO_ESTATE, "scratch too small for the fused functional pass");
    if ((rc = push_uex_table(p))) return rc;
    TriArgs A = tri_args(p, p->d_scratch);
    k_nlpoisson_p1_cell<OP_OUT_BOTH><<<grid_for(nc), kThreads, 0, p->stream>>>(A);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    if ((rc = segreduce(p, p->dvm_state[1], p->state.ndofs, d_dJdu))) return rc;
    const double *src = p->d_scratch + 3 * nc + (partitioned(p) ? p->cown_off : 0);
    const int64_t cnt = partitioned(p) ? p->cown_n : nc;
    const int g = red_grid(p, cnt);
    k_sum<<<g, kThreads, 0, p->stream>>>(src, cnt, p->d_partials);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    if ((rc = reduce_to(p, p->d_partials, nullptr, g, S_TMP1, 0))) return rc;
    return read_scalars(p, S_TMP1, 1, h_value);
}

// ---- linear algebra -------------------------------------------------------
int femo_spmv(femo_problem *p, int which, const double *d_vals, const double *d_x, double *d_y, int transpose) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (which < 0 || which > p->nin || !d_vals || !d_x || !d_y) return set_err(FEMO_EINVAL, "femo_spmv: bad arguments");
    const Pattern &P = p->pat[which];
    const DevPattern &D = p->dpat[which];
    // ghost refresh of the input: node vector for dR/du and for transposed dR/dm, cell vector for dR/dm
    if (which == 0 || transpose) {
        if ((rc = halo_nodes(p, const_cast<double *>(d_x)))) return rc;
    } else if ((rc = halo_cells(p, const_cast<double *>(d_x)))) return rc;
    if (!transpose) return launch_spmv<false>(p, D.rb, D.nrb, D.rowptr, D.col, d_vals, d_x, d_y, nullptr, nullptr, false);
    k_permute<<<grid_for(P.nnz), kThreads, 0, p->stream>>>(D.t_perm, d_vals, p->d_tvals, P.nnz);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return launch_spmv<false>(p, D.t_rb, D.t_nrb, D.t_rowptr, D.t_col, p->d_tvals, d_x, d_y, nullptr, nullptr, false);
}

/* y = A x with the dR/du values re-laid out as 3x3 blocks (BSR-3, K7 of SURVEY.md section 8a); convert != 0 refreshes
 * the block copy from d_vals first.  Only for states with 3 components per vertex (FEMO_ELIMIT otherwise). */
int femo_spmv_bsr3(femo_problem *p, const double *d_vals, const double *d_x, double *d_y, int convert) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_x || !d_y || (convert && !d_vals)) return set_err(FEMO_EINVAL, "femo_spmv_bsr3: null pointer");
    if (!p->dpat[0].b_perm || !p->d_bvals) return set_err(FEMO_ELIMIT, "femo_spmv_bsr3: the dR/du pattern is not made of complete 3x3 blocks");
    if (convert && (rc = bsr3_convert(p, d_vals))) return rc;
    return launch_spmv_bsr3<false>(p, d_x, d_y, nullptr, nullptr);
}

int femo_filter_apply3(int device, void *stream, int nx, int ny, int nz, double dx, double dy, double dz, double radius,
                       const double *d_in, double *d_out, double *d_den, int transpose) {
    if (nx < 1 || ny < 1 || nz < 1 || !(dx > 0) || !(dy > 0) || !(dz > 0) || !(radius > 0) || !d_in || !d_out || !d_den)
        return set_err(FEMO_EINVAL, "femo_filter_apply: bad arguments");
    if (femo_device_count() <= device || device < 0)
        return set_err(FEMO_ENODEVICE, "femo_filter_apply: no such CUDA device; this engine has no CPU path");
    FEMO_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)nx * ny * nz;
    const FilterLat L{nx, ny, nz, dx, dy, dz, radius};
    k_filter_den<<<grid_for(n), kThreads, 0, st>>>(L, d_den);
    if (transpose) k_filter_apply<true><<<grid_for(n), kThreads, 0, st>>>(L, d_den, d_in, d_out);
    else k_filter_apply<false><<<grid_for(n), kThreads, 0, st>>>(L, d_den, d_in, d_out);
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

int femo_filter_apply(int device, void *stream, int nx, int ny, double dx, double dy, double radius,
                      const double *d_in, double *d_out, double *d_den, int transpose) {
    return femo_filter_apply3(device, stream, nx, ny, 1, dx, dy, 1.0, radius, d_in, d_out, d_den, transpose);
}

int femo_pointwise_divide(femo_problem *p, double a, const double *d_num, const double *d_den, double *d_out, int64_t n) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_num || !d_den || !d_out || n < 0) return set_err(FEMO_EINVAL, "femo_pointwise_divide: bad arguments");
    k_divide<<<red_grid(p, n), kThreads, 0, p->stream>>>(a, d_num, d_den, d_out, n);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

int femo_axpy(femo_problem *p, double a, const double *d_x, double *d_y, int64_t n) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_x || !d_y || n < 0) return set_err(FEMO_EINVAL, "femo_axpy: bad arguments");
    k_axpy<<<red_grid(p, n), kThreads, 0, p->stream>>>(a, d_x, d_y, n);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

int femo_linear_solve(femo_problem *p, const double *d_vals, const double *d_b, double *d_x, int transpose,
                      const femo_krylov_opts *opts, femo_krylov_info *info) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_vals || !d_b || !d_x) return set_err(FEMO_EINVAL, "femo_linear_solve: null pointer");
    femo_krylov_opts o;
    memset(&o, 0, sizeof(o));
    if (opts) o = *opts;
    const double *vals = d_vals;
    if (transpose) {
        const int64_t nnz = p->pat[0].nnz;
        k_permute<<<grid_for(nnz), kThreads, 0, p->stream>>>(p->dpat[0].t_perm, d_vals, p->d_tvals, nnz);
        p->launches++;
        FEMO_CHECK_LAUNCH();
        vals = p->d_tvals;
    }
    return o.method == 1 ? gmres_solve(p, vals, d_b, d_x, o, info) : cg_solve(p, vals, d_b, d_x, o, info);
}

// ---------------------------------------------------------------------------------------------------------------
// Smoothed-aggregation AMG (precond 4): pattern phase on the host, arena handed in by the caller, numeric phase and
// V-cycle on the device (amg_setup.cpp, amg.cuh)
// ---------------------------------------------------------------------------------------------------------------
int femo_amg_symbolic(femo_problem *p, const double *h_vals, const femo_amg_opts *opts, int64_t info[4]) {
    if (!p) return set_err(FEMO_EINVAL, "femo_amg_symbolic: null problem");
    if (p->slab.active) return set_err(FEMO_ESTATE, "femo_amg_symbolic: slab problems use the lattice hierarchy");
    const Pattern &P = p->pat[0];
    if (P.nrows != P.ncols || P.nrows <= 0) return set_err(FEMO_ESTATE, "femo_amg_symbolic: no square state pattern");
    AmgOpts o;
    o.block = p->state.block;
    if (opts) {
        if (opts->theta >= 0.0) o.theta = opts->theta;
        if (opts->theta_decay > 0.0) o.theta_decay = opts->theta_decay;
        if (opts->max_levels > 0) o.max_levels = std::min(opts->max_levels, 24);
        if (opts->coarse_size > 0) o.coarse_size = std::min(opts->coarse_size, kMgDenseMax);
        if (opts->block > 0) o.block = opts->block;
        if (opts->omega_scale_set) o.omega_scale = opts->omega_scale;
    }
    delete p->amg;
    p->amg = new femo_amg();
    std::vector<uint8_t> iso;
    if ((p->has_bc && !p->bc_mark.empty()) || p->gpart.active) {
        // rows the coarse correction leaves alone: Dirichlet rows, and on a partition the ghost rows (below level 0 the
        // hierarchy is local to the rank, amg.cuh)
        iso.assign(P.nrows, 0);
        if (p->has_bc && !p->bc_mark.empty()) iso = p->bc_mark;
        if (p->gpart.active)
            for (int64_t r = p->gpart.n_owned_dofs; r < P.nrows; ++r) iso[r] = 1;
    }
    try {
        amg_build(P.rowptr.data(), P.col.data(), P.nrows, h_vals, iso.empty() ? nullptr : iso.data(), o, p->amg->host);
    } catch (const LayoutError &e) {
        delete p->amg;
        p->amg = nullptr;
        return set_err(e.code, e.msg);
    }
    Arena count;
    std::vector<AmgLevelDev> lv;
    amg_lay_out(count, p, p->amg->host, lv);
    p->amg->arena_bytes = count.used;
    if (info) {
        int64_t tot = 0;
        for (const AmgLevelHost &L : p->amg->host.lv) tot += L.nnz;
        info[0] = (int64_t)p->amg->host.lv.size();
        info[1] = (int64_t)p->amg->arena_bytes;
        info[2] = tot;
        info[3] = p->amg->host.lv.back().n;
    }
    return FEMO_OK;
}

int femo_amg_attach(femo_problem *p, void *d_arena, int64_t bytes) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!p->amg) return set_err(FEMO_ESTATE, "femo_amg_attach: run femo_amg_symbolic first");
    if (!d_arena || bytes < (int64_t)p->amg->arena_bytes) return set_err(FEMO_EINVAL, "femo_amg_attach: arena too small");
    return amg_attach(p, p->amg, d_arena, (size_t)bytes);
}

int femo_amg_numeric(femo_problem *p, const double *d_vals) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!d_vals) return set_err(FEMO_EINVAL, "femo_amg_numeric: null values");
    return amg_numeric(p, p->amg, d_vals);
}

int femo_amg_level_info(const femo_problem *p, int level, int64_t info[8], double dinfo[2]) {
    if (!p || !p->amg || level < 0 || level >= (int)p->amg->host.lv.size()) return set_err(FEMO_EINVAL, "femo_amg_level_info: no such level");
    const AmgLevelHost &L = p->amg->host.lv[level];
    if (info) {
        info[0] = L.n; info[1] = L.nnz; info[2] = L.nc; info[3] = L.nnzP; info[4] = L.nnzAP;
        info[5] = (int64_t)L.ap_ia.size(); info[6] = (int64_t)L.ac_ia.size(); info[7] = (int64_t)L.pp_src.size();
    }
    if (dinfo) {
        dinfo[0] = L.lmax;                                                           // host numeric phase
        dinfo[1] = (p->amg->attached && level < (int)p->amg->lv.size()) ? p->amg->lv[level].lmax : 0.0;   // device numeric phase
    }
    return FEMO_OK;
}

int femo_amg_level_array(const femo_problem *p, int level, int which, int32_t *h_out, int64_t cap) {
    if (!p || !p->amg || level < 0 || level >= (int)p->amg->host.lv.size()) return set_err(FEMO_EINVAL, "femo_amg_level_array: no such level");
    const AmgLevelHost &L = p->amg->host.lv[level];
    const std::vector<int32_t> *v[] = {&L.rowptr, &L.col, &L.agg, &L.p_rowptr, &L.p_col, &L.pp_ptr, &L.pp_src, &L.r_rowptr, &L.r_col,
                                       &L.r_perm, &L.ap_rowptr, &L.ap_col, &L.ap_ptr, &L.ap_ia, &L.ap_ib, &L.ac_ptr, &L.ac_ia, &L.ac_ib};
    if (which < 0 || which >= (int)(sizeof(v) / sizeof(v[0]))) return set_err(FEMO_EINVAL, "femo_amg_level_array: which 0..17");
    if (!h_out || cap < (int64_t)v[which]->size()) return set_err(FEMO_EINVAL, "femo_amg_level_array: output too small");
    if (!v[which]->empty()) memcpy(h_out, v[which]->data(), v[which]->size() * sizeof(int32_t));
    return (int)FEMO_OK;
}

int femo_amg_level_values(femo_problem *p, int level, int which, int from_device, double *h_out, int64_t cap) {
    if (!p || !p->amg || level < 0 || level >= (int)p->amg->host.lv.size()) return set_err(FEMO_EINVAL, "femo_amg_level_values: no such level");
    const AmgLevelHost &L = p->amg->host.lv[level];
    if (which < 0 || which > 3) return set_err(FEMO_EINVAL, "femo_amg_level_values: which 0 operator, 1 prolongator, 2 A*P, 3 inverse diagonal");
    const int64_t len = which == 0 ? L.nnz : which == 1 ? L.nnzP : which == 2 ? L.nnzAP : L.n;
    if (!h_out || cap < len) return set_err(FEMO_EINVAL, "femo_amg_level_values: output too small");
    if (!from_device) {
        const std::vector<double> &v = which == 0 ? L.vals : which == 1 ? L.p_vals : which == 2 ? L.ap_vals : L.dinv;
        if ((int64_t)v.size() != len) return set_err(FEMO_ESTATE, "femo_amg_level_values: the hierarchy was built from the pattern only (no host values)");
        if (len) memcpy(h_out, v.data(), len * sizeof(double));
        return FEMO_OK;
    }
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!p->amg->attached || !p->amg->numeric_setups) return set_err(FEMO_ESTATE, "femo_amg_level_values: no numeric phase has run on the device");
    const AmgLevelDev &D = p->amg->lv[level];
    const double *src = which == 0 ? D.vals : which == 1 ? D.p_vals : which == 2 ? D.ap_vals : D.dinv;
    if (!src) return set_err(FEMO_ESTATE, "femo_amg_level_values: array does not exist on this level");
    FEMO_CUDA(cudaStreamSynchronize(p->stream));
    FEMO_CUDA(cudaMemcpy(h_out, src, len * sizeof(double), cudaMemcpyDeviceToHost));
    return FEMO_OK;
}

/* measurement hook (bench.py roofline): ONE launch of the fine-level V-cycle operator kernel in `mode`
 * (0 residual, 1 first / 2 later Chebyshev step, 3 fused zero-guess pre-smoother, 6 / 7 down / up level sweep) on the
 * hierarchy the last multigrid-preconditioned solve set up; vectors are the solver's own work vectors.  info[0] =
 * algorithmic bytes of the launch, info[1] = fine-level launches of this mode so far (before this one). */
int femo_vcycle_op_probe(femo_problem *p, int mode, int64_t info[2]) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (mode < 0 || mode > 7) return set_err(FEMO_EINVAL, "femo_vcycle_op_probe: mode 0..7");
    if (!dia_ready(p)) return set_err(FEMO_ESTATE, "femo_vcycle_op_probe: no DIA hierarchy (run a precond=2 solve on a lattice P1 problem first)");
    const int64_t N = p->state.ndofs;
    if (mode >= 6) {
        // down: b, dinv, 7 planes read, x_pre written, coarse b written ; up: x_pre, b, 7 planes + dinv read, coarse x read,
        // x written ; + the Dirichlet marks read once when the level has them
        const MgParams mp;
        if (p->mg.empty() || !mgsweep_ok(p, p->mg[0], mp))
            return set_err(FEMO_ESTATE, "femo_vcycle_op_probe: the fine level does not take the level sweeps");
        femo_problem *C = p->mg[0];
        const int64_t nc = C->state.ndofs;
        int64_t bytes = mode == 6 ? 48 * N + 8 * nc : 56 * N + 8 * nc;
        if (p->has_bc) bytes += N;
        if (mode == 6 && C->has_bc) bytes += nc;
        if (info) { info[0] = bytes; info[1] = p->sweep_count[mode - 6]; }
        return mode == 6 ? mgsweep_down(p, C, p->kr_r, p->kr_d, mp) : mgsweep_up(p, C, p->kr_r, p->kr_d, p->kr_z, mp);
    }
    if (mode >= 4) {
        // fp64 planes of the CG recurrence: 7 x 8 B values + x read + y written; mode 4 = fused dot(x, y), 5 = plain
        if (!p->mgl.dia64) return set_err(FEMO_ESTATE, "femo_vcycle_op_probe: no fp64 DIA planes on this problem");
        if (info) { info[0] = 72 * N; info[1] = p->dia64_count[mode - 4]; }
        return mode == 4 ? launch_dia64<true>(p, p->kr_d, p->kr_w, nullptr, nullptr) : launch_dia64<false>(p, p->kr_d, p->kr_w, nullptr, nullptr);
    }
    DiaEpi E;
    E.b = p->kr_r; E.rin = p->kr_r; E.c0 = 0.5; E.c1 = 0.25; E.c2 = 0.125;
    int64_t bytes = 28 * N;                                   // 7 fp32 planes
    if (mode == DIA_PLAIN) bytes += 24 * N;                   // x, b read; r written
    if (mode == DIA_CHEB0) { E.rout = p->kr_w; E.dout = p->kr_q; bytes += 36 * N; }     // scaling plane; x, b read; r, d written
    if (mode == DIA_CHEBK) { E.xacc = p->kr_z; E.xmode = 0; bytes += 36 * N; }          // scaling plane; d, r read; x read + written
    if (mode == DIA_PRE2) bytes += 20 * N;                    // scaling plane; b read; x written
    if (info) { info[0] = bytes; info[1] = p->dia_count[mode]; }
    return launch_dia(p, mode, p->kr_d, mode == DIA_PRE2 ? p->kr_z : p->kr_w, E);
}

int femo_newton_solve(femo_problem *p, const femo_newton_opts *opts, femo_newton_info *info) {
    int rc;
    if ((rc = need_device(p))) return rc;
    if (!opts) return set_err(FEMO_EINVAL, "femo_newton_solve: null options");
    if ((rc = need_coef(p, 0, p->state.ndofs, "state"))) return rc;
    const int64_t n = p->state.ndofs;
    double *x = const_cast<double *>(p->coef[0]);  // the state slot is updated in place
    cudaStream_t st = p->stream;
    const bool snes = opts->kind == 1;
    double *vals_bc = p->has_bc ? p->nt_vals_bc : p->nt_vals;
    int it = 0, kit = 0, spmvs = 0, reason = 0;
    double f0 = 0, fn = 0, f_prev = 0, eta_prev = 0;
    bool jac_valid = false;
    // lattice P1 problems solved by GMG-PCG: the Jacobian rows go straight into the DIA planes of the solve
    const bool lat_direct = opts->krylov.precond == 2 && opts->krylov.mg_precision == 0 && opts->krylov.method == 0 &&
                            !p->mg.empty() && lattice_dia_direct(p);
    p->mgl.dinv = p->kr_dinv;
    auto eval_F = [&]() -> int {
        int r;
        jac_valid = false;
        if (p->has_bc) {  // lifting needs the element columns of Dirichlet dofs at this state
            if (lat_direct) r = lattice_jacobian(p, p->nt_vals, p->nt_vals_bc, true, true);
            else r = femo_assemble_jacobian(p, p->nt_vals, p->nt_vals_bc);
            if (r) return r;
            jac_valid = true;
        }
        if ((r = femo_newton_rhs(p, p->nt_vals, p->nt_b))) return r;
        double s;
        if ((r = norm2_sq(p, p->nt_b, &s))) return r;
        fn = std::sqrt(s);
        return FEMO_OK;
    };
    if ((rc = eval_F())) return rc;
    f0 = fn;
    if (fn < opts->atol) reason = 1;
    while (!reason && it < opts->max_it) {
        if (!jac_valid && (rc = lat_direct ? lattice_jacobian(p, nullptr, nullptr, true, false)   // no CSR copy needed
                                           : femo_assemble_jacobian(p, p->nt_vals, nullptr))) return rc;
        k_fill<<<red_grid(p, n), kThreads, 0, st>>>(0.0, p->nt_dx, n);
        p->launches++;
        femo_krylov_info ki;
        memset(&ki, 0, sizeof(ki));
        // inexact Newton: a linear residual below a tenth of the nonlinear absolute tolerance cannot
        // change the SNES convergence decision, so the Krylov solve may stop there
        femo_krylov_opts ko = opts->krylov;
        if (snes) ko.atol = std::max(ko.atol, 0.1 * opts->atol);
        if (opts->krylov.forcing > 0.0) {
            // Eisenstat-Walker forcing (choice 2, gamma 0.9, alpha 2, with their safeguard): the linear tolerance follows
            // the observed nonlinear contraction, never looser than `forcing`, never tighter than the caller's rtol
            double eta = opts->krylov.forcing;
            if (it > 0 && f_prev > 0.0) {
                eta = 0.9 * (fn / f_prev) * (fn / f_prev);
                const double guard = 0.9 * eta_prev * eta_prev;
                if (guard > 0.1) eta = std::max(eta, guard);
                eta = std::min(eta, opts->krylov.forcing);
            }
            ko.rtol = std::max(eta, opts->krylov.rtol > 0 ? opts->krylov.rtol : 1e-10);
            eta_prev = ko.rtol;
        }
        f_prev = fn;
        if ((rc = (ko.method == 1 ? gmres_solve(p, vals_bc, p->nt_b, p->nt_dx, ko, &ki) : cg_solve(p, vals_bc, p->nt_b, p->nt_dx, ko, &ki, true, lat_direct)))) return rc;
        kit += ki.iterations;
        spmvs += ki.spmv_count;
        // the reference's LU cannot fail; a Krylov solve can (max_it, breakdown, NaN): never apply such a step silently
        if (!ki.converged || !(ki.rnorm == ki.rnorm)) {
            if (info) {
                info->iterations = it; info->converged = -1; info->fnorm0 = f0; info->fnorm = fn;
                info->krylov_iterations = kit; info->spmv_count = spmvs;
            }
            return set_err(FEMO_ENOCONV, "linear solve inside the Newton iteration did not converge (Krylov max_it reached or non-finite residual)");
        }
        k_axpy<<<red_grid(p, n), kThreads, 0, st>>>(-1.0, p->nt_dx, x, n);
        p->launches++;
        FEMO_CHECK_LAUNCH();
        if ((rc = eval_F())) return rc;
        ++it;
        if (!(fn == fn) || std::isinf(fn)) return set_err(FEMO_ENOCONV, "Newton iteration produced a non-finite residual norm");
        if (fn < opts->atol) reason = 1;
        else if (snes ? (fn <= opts->rtol * f0) : (f0 > 0 && fn / f0 < opts->rtol)) reason = 2;
        else if (snes) {
            double sy, sx;
            if ((rc = norm2_sq(p, p->nt_dx, &sy))) return rc;
            if ((rc = norm2_sq(p, x, &sx))) return rc;
            if (std::sqrt(sy) < opts->stol * std::sqrt(sx)) reason = 3;
        }
    }
    if (info) {
        info->iterations = it;
        info->converged = reason;
        info->fnorm0 = f0;
        info->fnorm = fn;
        info->krylov_iterations = kit;
        info->spmv_count = spmvs;
    }
    if (snes && !reason) return set_err(FEMO_ENOCONV, "SNES did not converge within max_it");
    return FEMO_OK;
}

}  // extern "C"
