// multigrid.cuh -- geometric multigrid preconditioner for vertex-based spaces on
// lattice meshes, used by the Krylov drivers in place of the reference's direct
// LU (KSP preonly + PC lu/MUMPS, femo/fea/utils_dolfinx.py:405-408,476-512).
//
//   * levels: the lattice is halved (ceil) per direction until <= kMgCoarsest
//     cells; levels need not be nested -- transfers evaluate the coarse P1
//     basis at the fine nodes (matrix-free, R = P^T by construction)
//   * coarse operators: rediscretised with the family's own Jacobian kernel on
//     the coarse mesh, state interpolated to the coarse nodes, Dirichlet rows
//     inherited geometrically
//   * smoother: Chebyshev polynomial on the Jacobi-scaled operator, eigenvalue
//     bound by Gershgorin (deterministic, no power iteration), same polynomial
//     before and after the coarse correction => symmetric preconditioner for CG
//   * coarsest level: explicit inverse computed by one CTA (Gauss-Jordan)
//
// Included by engine.cu (single translation unit).
#pragma once
#include "common.cuh"

namespace femo {

constexpr int kMgCoarsest = 8;      // stop coarsening a direction at <= 8 cells
constexpr int kMgDenseMax = 512;    // largest coarsest-level system inverted explicitly

struct Lattice {
    int nx, ny;  // cells per direction; nodes are (nx+1) x (ny+1), node id = j*(nx+1)+i
};

// P1 hat function of a node of the "right"-diagonal triangulation, lattice units
__device__ __forceinline__ double hat_p1(double dx, double dy) {
    const double v = 1.0 - fmax(fmax(dx, dy), 0.0) + fmin(fmin(dx, dy), 0.0);
    return v > 0.0 ? v : 0.0;
}

// bilinear Q1 hat on the tensor lattice
__device__ __forceinline__ double hat_q1(double dx, double dy) {
    const double a = 1.0 - fabs(dx), b = 1.0 - fabs(dy);
    return (a > 0.0 && b > 0.0) ? a * b : 0.0;
}
__device__ __forceinline__ double hat_of(int kind, double dx, double dy) { return kind ? hat_q1(dx, dy) : hat_p1(dx, dy); }

// vector loads of the transfer bodies: CG = true reads through L2 only (ld.global.cg) -- used by the fused cooperative
// V-cycle kernel, where the vector was written earlier in the SAME kernel by other SMs
template <bool CG>
__device__ __forceinline__ double ldv(const double *p) { return CG ? __ldcg(p) : *p; }

// dst(dof) (+)= sum_k phi^src_k(x_node) src(k): prolongation (src = coarse) and state interpolation
// (src = fine) share this body.  `block` interleaved components per node, hat 0 = P1 right-diagonal, 1 = Q1.
template <bool ADD, bool CG = false>
__device__ __forceinline__ void lattice_interp_at(Lattice s, Lattice d, int block, int hat, const double *src, double *dst,
                                                  const uint8_t *dst_mask, int64_t idx) {
    if (dst_mask && dst_mask[idx]) {
        if (!ADD) dst[idx] = 0.0;
        return;
    }
    const int64_t node = idx / block;
    const int comp = (int)(idx % block);
    const int i = (int)(node % (d.nx + 1)), j = (int)(node / (d.nx + 1));
    const double X = (double)i * ((double)s.nx / (double)d.nx), Y = (double)j * ((double)s.ny / (double)d.ny);
    const int I = min((int)X, s.nx - 1), J = min((int)Y, s.ny - 1);
    double acc = 0.0;
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const double w = hat_of(hat, X - (double)(I + a), Y - (double)(J + b));
            if (w > 0.0) acc += w * ldv<CG>(src + ((int64_t)(J + b) * (s.nx + 1) + (I + a)) * block + comp);
        }
    if (ADD) dst[idx] = ldv<CG>(dst + idx) + acc;
    else dst[idx] = acc;
}

template <bool ADD>
__global__ void __launch_bounds__(kThreads)
    k_lattice_interp(Lattice s, Lattice d, int block, int hat, const double *__restrict__ src, double *__restrict__ dst,
                     const uint8_t *__restrict__ dst_mask) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nd = (int64_t)(d.nx + 1) * (d.ny + 1) * block;
    if (idx >= nd) return;
    lattice_interp_at<ADD>(s, d, block, hat, src, dst, dst_mask, idx);
}

// rc = P^T rf with the same weights as lattice_interp_at<coarse -> fine>
template <bool CG = false>
__device__ __forceinline__ void lattice_restrict_at(Lattice f, Lattice c, int block, int hat, const double *rf, double *rc,
                                                    const uint8_t *mask_f, const uint8_t *mask_c, int64_t idx) {
    if (mask_c && mask_c[idx]) {
        rc[idx] = 0.0;
        return;
    }
    const int64_t node = idx / block;
    const int comp = (int)(idx % block);
    const int I = (int)(node % (c.nx + 1)), J = (int)(node / (c.nx + 1));
    const double sx = (double)c.nx / (double)f.nx, sy = (double)c.ny / (double)f.ny;
    const int ilo = max(0, (int)floor((double)(I - 1) / sx)), ihi = min(f.nx, (int)ceil((double)(I + 1) / sx));
    const int jlo = max(0, (int)floor((double)(J - 1) / sy)), jhi = min(f.ny, (int)ceil((double)(J + 1) / sy));
    double acc = 0.0;
    for (int j = jlo; j <= jhi; ++j)
        for (int i = ilo; i <= ihi; ++i) {
            // the fine node must see (I,J) as a corner of its enclosing coarse cell, as the prolongation does
            const double X = (double)i * sx, Y = (double)j * sy;
            const int I0 = min((int)X, c.nx - 1), J0 = min((int)Y, c.ny - 1);
            if (I < I0 || I > I0 + 1 || J < J0 || J > J0 + 1) continue;
            const double w = hat_of(hat, X - (double)I, Y - (double)J);
            const int64_t fi = ((int64_t)j * (f.nx + 1) + i) * block + comp;
            if (w > 0.0 && !(mask_f && mask_f[fi])) acc += w * ldv<CG>(rf + fi);
        }
    rc[idx] = acc;
}

__global__ void __launch_bounds__(kThreads)
    k_lattice_restrict(Lattice f, Lattice c, int block, int hat, const double *__restrict__ rf, double *__restrict__ rc,
                       const uint8_t *__restrict__ mask_f, const uint8_t *__restrict__ mask_c) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nc = (int64_t)(c.nx + 1) * (c.ny + 1) * block;
    if (idx >= nc) return;
    lattice_restrict_at(f, c, block, hat, rf, rc, mask_f, mask_c, idx);
}

// coarse cell-wise coefficient for the rediscretised SIMP operator: power mean of the fine densities whose
// cell centres lie in the coarse cell, rho_c = (mean rho_f^p)^(1/p)  (quadrilateral lattices, one value per cell)
__global__ void __launch_bounds__(kThreads)
    k_restrict_cells_power(Lattice f, Lattice c, double p, const double *__restrict__ rf, double *__restrict__ rc) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)c.nx * c.ny) return;
    const int I = (int)(idx % c.nx), J = (int)(idx / c.nx);
    const int i0 = (int)ceil(((double)I * f.nx) / c.nx - 0.5), i1 = (int)ceil(((double)(I + 1) * f.nx) / c.nx - 0.5);
    const int j0 = (int)ceil(((double)J * f.ny) / c.ny - 0.5), j1 = (int)ceil(((double)(J + 1) * f.ny) / c.ny - 0.5);
    double acc = 0.0;
    int cnt = 0;
    for (int j = max(j0, 0); j < min(j1, f.ny); ++j)
        for (int i = max(i0, 0); i < min(i1, f.nx); ++i) {
            acc += pow(rf[(int64_t)j * f.nx + i], p);
            ++cnt;
        }
    rc[idx] = cnt ? pow(acc / cnt, 1.0 / p) : 1.0;
}

// ---- hexahedral lattices (trilinear Q1), same conventions in three dimensions ---------------------
struct Lattice3 {
    int nx, ny, nz;  // cells per direction; node id = (k*(ny+1)+j)*(nx+1)+i
};
static inline Lattice3 lat3_of(const Mesh &m) { return Lattice3{m.n[0], m.n[1], m.n[2]}; }

__device__ __forceinline__ double hat_1d(double d) {
    const double a = 1.0 - fabs(d);
    return a > 0.0 ? a : 0.0;
}

template <bool ADD>
__global__ void __launch_bounds__(kThreads)
    k_lattice3_interp(Lattice3 s, Lattice3 d, int block, const double *__restrict__ src, double *__restrict__ dst,
                      const uint8_t *__restrict__ dst_mask) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nd = (int64_t)(d.nx + 1) * (d.ny + 1) * (d.nz + 1) * block;
    if (idx >= nd) return;
    if (dst_mask && dst_mask[idx]) {
        if (!ADD) dst[idx] = 0.0;
        return;
    }
    const int64_t node = idx / block;
    const int comp = (int)(idx % block);
    const int i = (int)(node % (d.nx + 1)), j = (int)((node / (d.nx + 1)) % (d.ny + 1)), k = (int)(node / ((int64_t)(d.nx + 1) * (d.ny + 1)));
    const double X = (double)i * ((double)s.nx / (double)d.nx), Y = (double)j * ((double)s.ny / (double)d.ny),
                 Z = (double)k * ((double)s.nz / (double)d.nz);
    const int I = min((int)X, s.nx - 1), J = min((int)Y, s.ny - 1), K = min((int)Z, s.nz - 1);
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
            for (int a = 0; a < 2; ++a) {
                const double w = hat_1d(X - (double)(I + a)) * hat_1d(Y - (double)(J + b)) * hat_1d(Z - (double)(K + c));
                if (w > 0.0) acc += w * src[(((int64_t)(K + c) * (s.ny + 1) + (J + b)) * (s.nx + 1) + (I + a)) * block + comp];
            }
    if (ADD) dst[idx] += acc;
    else dst[idx] = acc;
}

// rc = P^T rf with the weights of k_lattice3_interp<coarse -> fine>
__global__ void __launch_bounds__(kThreads)
    k_lattice3_restrict(Lattice3 f, Lattice3 c, int block, const double *__restrict__ rf, double *__restrict__ rc,
                        const uint8_t *__restrict__ mask_f, const uint8_t *__restrict__ mask_c) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nc = (int64_t)(c.nx + 1) * (c.ny + 1) * (c.nz + 1) * block;
    if (idx >= nc) return;
    if (mask_c && mask_c[idx]) {
        rc[idx] = 0.0;
        return;
    }
    const int64_t node = idx / block;
    const int comp = (int)(idx % block);
    const int I = (int)(node % (c.nx + 1)), J = (int)((node / (c.nx + 1)) % (c.ny + 1)), K = (int)(node / ((int64_t)(c.nx + 1) * (c.ny + 1)));
    const double sx = (double)c.nx / (double)f.nx, sy = (double)c.ny / (double)f.ny, sz = (double)c.nz / (double)f.nz;
    const int ilo = max(0, (int)floor((double)(I - 1) / sx)), ihi = min(f.nx, (int)ceil((double)(I + 1) / sx));
    const int jlo = max(0, (int)floor((double)(J - 1) / sy)), jhi = min(f.ny, (int)ceil((double)(J + 1) / sy));
    const int klo = max(0, (int)floor((double)(K - 1) / sz)), khi = min(f.nz, (int)ceil((double)(K + 1) / sz));
    double acc = 0.0;
    for (int k = klo; k <= khi; ++k) {
        const double Z = (double)k * sz;
        const int K0 = min((int)Z, c.nz - 1);
        if (K < K0 || K > K0 + 1) continue;
        const double wz = hat_1d(Z - (double)K);
        for (int j = jlo; j <= jhi; ++j) {
            const double Y = (double)j * sy;
            const int J0 = min((int)Y, c.ny - 1);
            if (J < J0 || J > J0 + 1) continue;
            const double wy = hat_1d(Y - (double)J);
            for (int i = ilo; i <= ihi; ++i) {
                const double X = (double)i * sx;
                const int I0 = min((int)X, c.nx - 1);
                if (I < I0 || I > I0 + 1) continue;
                const double w = hat_1d(X - (double)I) * wy * wz;
                const int64_t fi = (((int64_t)k * (f.ny + 1) + j) * (f.nx + 1) + i) * block + comp;
                if (w > 0.0 && !(mask_f && mask_f[fi])) acc += w * rf[fi];
            }
        }
    }
    rc[idx] = acc;
}

__global__ void __launch_bounds__(kThreads)
    k_restrict_cells_power3(Lattice3 f, Lattice3 c, double p, const double *__restrict__ rf, double *__restrict__ rc) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)c.nx * c.ny * c.nz) return;
    const int I = (int)(idx % c.nx), J = (int)((idx / c.nx) % c.ny), K = (int)(idx / ((int64_t)c.nx * c.ny));
    const int i0 = (int)ceil(((double)I * f.nx) / c.nx - 0.5), i1 = (int)ceil(((double)(I + 1) * f.nx) / c.nx - 0.5);
    const int j0 = (int)ceil(((double)J * f.ny) / c.ny - 0.5), j1 = (int)ceil(((double)(J + 1) * f.ny) / c.ny - 0.5);
    const int k0 = (int)ceil(((double)K * f.nz) / c.nz - 0.5), k1 = (int)ceil(((double)(K + 1) * f.nz) / c.nz - 0.5);
    double acc = 0.0;
    int cnt = 0;
    for (int k = max(k0, 0); k < min(k1, f.nz); ++k)
        for (int j = max(j0, 0); j < min(j1, f.ny); ++j)
            for (int i = max(i0, 0); i < min(i1, f.nx); ++i) {
                acc += pow(rf[((int64_t)k * f.ny + j) * f.nx + i], p);
                ++cnt;
            }
    rc[idx] = cnt ? pow(acc / cnt, 1.0 / p) : 1.0;
}

// 2:1 nested lattices (the common case), integer-only, slab aware.  A local lattice holds node rows
// [j0, j0+nrows) of the global lattice; prolongation / restriction / injection address the other
// level through GLOBAL row indices, so the same kernels serve one GPU (j0 = 0), two distributed
// slabs, and a distributed fine level over a replicated coarse level.  Rows that would need data
// outside the local slab are ghost rows: they are skipped / partial and refreshed by halo exchange.
struct LatD {
    int nx, nrows, j0;
};

// value-level expressions of the nested transfers, shared with the fused level sweeps (mgsweep.cuh)
// xf + P xc at a fine node: a = xc at the coarse node (i>>1, j>>1), a2 = xc at (+oi, +oj); odd = oi | oj
__device__ __forceinline__ double prolong_nested_val(double xf, double a, double a2, bool odd) {
    return xf + (odd ? 0.5 * (a + a2) : a);
}
// P^T r at a coarse node from the fine residual at the coincident node c and its six stencil neighbours (left to right)
__device__ __forceinline__ double restrict_nested_val(double c, double l, double r, double d, double u, double dl, double ur) {
    return c + 0.5 * (l + r + d + u + dl + ur);
}

// weights of the right-diagonal P1 hat: 1 at coincident nodes, 1/2 along x, y and the (1,1) diagonal
template <bool CG = false>
__device__ __forceinline__ void prolong_nested_at(LatD f, LatD c, const double *xc, double *xf, const uint8_t *mask_f, int64_t idx) {
    const int fw = f.nx + 1, cw = c.nx + 1;
    if (mask_f && mask_f[idx]) return;
    const int i = (int)(idx % fw), jl = (int)(idx / fw);
    const int gj = jl + f.j0;
    const int I = i >> 1, oi = i & 1, oj = gj & 1;
    const int Jl = (gj >> 1) - c.j0;
    if (Jl < 0 || Jl + oj >= c.nrows) return;
    const double a = ldv<CG>(xc + (int64_t)Jl * cw + I);
    const double a2 = (oi | oj) ? ldv<CG>(xc + (int64_t)(Jl + oj) * cw + (I + oi)) : 0.0;
    xf[idx] = prolong_nested_val(ldv<CG>(xf + idx), a, a2, oi | oj);
}

__global__ void __launch_bounds__(kThreads)
    k_prolong_nested(LatD f, LatD c, const double *__restrict__ xc, double *__restrict__ xf,
                     const uint8_t *__restrict__ mask_f) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)(f.nx + 1) * f.nrows) return;
    prolong_nested_at(f, c, xc, xf, mask_f, idx);
}

template <bool CG = false>
__device__ __forceinline__ void restrict_nested_at(LatD f, LatD c, const double *rf, double *rc, const uint8_t *mask_f,
                                                   const uint8_t *mask_c, int64_t idx) {
    const int cw = c.nx + 1, fw = f.nx + 1;
    if (mask_c && mask_c[idx]) {
        rc[idx] = 0.0;
        return;
    }
    const int I = (int)(idx % cw), Jl = (int)(idx / cw);
    const int i = 2 * I, j = 2 * (Jl + c.j0) - f.j0;      // fine LOCAL row of the coincident node
    auto at = [&](int ii, int jj) -> double {
        if (ii < 0 || jj < 0 || ii > f.nx || jj >= f.nrows) return 0.0;
        const int64_t k = (int64_t)jj * fw + ii;
        return (mask_f && mask_f[k]) ? 0.0 : ldv<CG>(rf + k);
    };
    rc[idx] = restrict_nested_val(at(i, j), at(i - 1, j), at(i + 1, j), at(i, j - 1), at(i, j + 1), at(i - 1, j - 1), at(i + 1, j + 1));
}

__global__ void __launch_bounds__(kThreads)
    k_restrict_nested(LatD f, LatD c, const double *__restrict__ rf, double *__restrict__ rc,
                      const uint8_t *__restrict__ mask_f, const uint8_t *__restrict__ mask_c) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)(c.nx + 1) * c.nrows) return;
    restrict_nested_at(f, c, rf, rc, mask_f, mask_c, idx);
}

// coarse state = fine state at the coincident nodes (rediscretisation of the coarse Jacobian)
__global__ void __launch_bounds__(kThreads)
    k_inject_nested(LatD f, LatD c, const double *__restrict__ uf, double *__restrict__ uc) {
    const int cw = c.nx + 1, fw = f.nx + 1;
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)cw * c.nrows) return;
    const int I = (int)(idx % cw), Jl = (int)(idx / cw);
    const int j = 2 * (Jl + c.j0) - f.j0;
    uc[idx] = (j >= 0 && j < f.nrows) ? uf[(int64_t)j * fw + 2 * I] : 0.0;
}

// ---- the same three kernels for 2:1 nested hexahedral lattices cut into z-slabs (trilinear weights) ----------
struct LatD3 {
    int nx, ny, nplanes, k0;   // cells in x / y, local node planes, global index of local plane 0
};

__global__ void __launch_bounds__(kThreads)
    k_prolong_nested3(LatD3 f, LatD3 c, int block, const double *__restrict__ xc, double *__restrict__ xf,
                      const uint8_t *__restrict__ mask_f) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int fw = f.nx + 1, fh = f.ny + 1, cw = c.nx + 1, ch = c.ny + 1;
    if (idx >= (int64_t)fw * fh * f.nplanes * block) return;
    if (mask_f && mask_f[idx]) return;
    const int comp = (int)(idx % block);
    const int64_t node = idx / block;
    const int i = (int)(node % fw), j = (int)((node / fw) % fh), kl = (int)(node / ((int64_t)fw * fh));
    const int gk = kl + f.k0;
    const int I = i >> 1, oi = i & 1, J = j >> 1, oj = j & 1, ok = gk & 1;
    const int Kl = (gk >> 1) - c.k0;
    if (Kl < 0 || Kl + ok >= c.nplanes) return;
    double acc = 0.0;
    for (int d = 0; d <= ok; ++d)
        for (int b = 0; b <= oj; ++b)
            for (int a = 0; a <= oi; ++a) acc += xc[((((int64_t)(Kl + d) * ch) + (J + b)) * cw + (I + a)) * block + comp];
    const double w = 1.0 / (double)((1 + oi) * (1 + oj) * (1 + ok));
    xf[idx] += w * acc;
}

__global__ void __launch_bounds__(kThreads)
    k_restrict_nested3(LatD3 f, LatD3 c, int block, const double *__restrict__ rf, double *__restrict__ rc,
                       const uint8_t *__restrict__ mask_f, const uint8_t *__restrict__ mask_c) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int fw = f.nx + 1, fh = f.ny + 1, cw = c.nx + 1, ch = c.ny + 1;
    if (idx >= (int64_t)cw * ch * c.nplanes * block) return;
    if (mask_c && mask_c[idx]) {
        rc[idx] = 0.0;
        return;
    }
    const int comp = (int)(idx % block);
    const int64_t node = idx / block;
    const int I = (int)(node % cw), J = (int)((node / cw) % ch), Kl = (int)(node / ((int64_t)cw * ch));
    const int i = 2 * I, j = 2 * J, k = 2 * (Kl + c.k0) - f.k0;   // fine LOCAL plane of the coincident node
    double acc = 0.0;
    for (int dk = -1; dk <= 1; ++dk) {
        const int kk = k + dk;
        if (kk < 0 || kk >= f.nplanes) continue;
        for (int dj = -1; dj <= 1; ++dj) {
            const int jj = j + dj;
            if (jj < 0 || jj > f.ny) continue;
            for (int di = -1; di <= 1; ++di) {
                const int ii = i + di;
                if (ii < 0 || ii > f.nx) continue;
                const int64_t q = ((((int64_t)kk * fh) + jj) * fw + ii) * block + comp;
                if (mask_f && mask_f[q]) continue;
                acc += rf[q] * ((di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0));
            }
        }
    }
    rc[idx] = acc;
}

__global__ void __launch_bounds__(kThreads)
    k_inject_nested3(LatD3 f, LatD3 c, int block, const double *__restrict__ uf, double *__restrict__ uc) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int fw = f.nx + 1, fh = f.ny + 1, cw = c.nx + 1, ch = c.ny + 1;
    if (idx >= (int64_t)cw * ch * c.nplanes * block) return;
    const int comp = (int)(idx % block);
    const int64_t node = idx / block;
    const int I = (int)(node % cw), J = (int)((node / cw) % ch), Kl = (int)(node / ((int64_t)cw * ch));
    const int k = 2 * (Kl + c.k0) - f.k0;
    uc[idx] = (k >= 0 && k < f.nplanes) ? uf[((((int64_t)k * fh) + 2 * J) * fw + 2 * I) * block + comp] : 0.0;
}

// power-mean coarse density on 2:1 nested slabs: coarse local cell layer Kl <- fine local layers 2(Kl+ck0)-fk0, +1;
// layers outside the local slab are skipped (the ghost layer is refreshed by halo_cells afterwards)
__global__ void __launch_bounds__(kThreads)
    k_restrict_cells_power_nested3(int cnx, int cny, int cnl, int ck0, int fnl, int fk0, double p, const double *__restrict__ rf,
                                   double *__restrict__ rc) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)cnx * cny * cnl) return;
    const int I = (int)(idx % cnx), J = (int)((idx / cnx) % cny), Kl = (int)(idx / ((int64_t)cnx * cny));
    const int fnx = 2 * cnx, fny = 2 * cny, k = 2 * (Kl + ck0) - fk0;
    double acc = 0.0;
    int cnt = 0;
    for (int d = 0; d < 2; ++d) {
        if (k + d < 0 || k + d >= fnl) continue;
        for (int b = 0; b < 2; ++b)
            for (int a = 0; a < 2; ++a) {
                acc += pow(rf[((int64_t)(k + d) * fny + (2 * J + b)) * fnx + (2 * I + a)], p);
                ++cnt;
            }
    }
    rc[idx] = cnt ? pow(acc / cnt, 1.0 / p) : 1.0;
}

// Gershgorin bound of D^-1 A (max_i sum_j |a_ij| / |a_ii|) and dinv in one pass
__global__ void __launch_bounds__(kThreads)
    k_diag_gershgorin(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ vals,
                      double *__restrict__ dinv, int64_t n, int64_t o0, int64_t o1, double *__restrict__ partials) {
    double mx = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double d = 1.0, s = 0.0;
        for (int32_t t = rowptr[i]; t < rowptr[i + 1]; ++t) {
            const double v = vals[t];
            s += fabs(v);
            if (col[t] == i) d = v;
        }
        const double di = (d != 0.0) ? 1.0 / d : 1.0;
        dinv[i] = di;
        if (i >= o0 && i < o1) mx = fmax(mx, s * fabs(di));
    }
    // block max
    __shared__ double sh[kThreads];
    sh[threadIdx.x] = mx;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(kThreads) k_max_finalize(const double *__restrict__ partials, int np, double *scalars, int slot) {
    __shared__ double sh[kThreads];
    // four independent loads in flight per thread: the node-centric Jacobian hands over one partial per CTA (62 k of them
    // at n=4000) and a single dependent chain of L2 loads took 114 us (ncu launch list r3n); max is order-independent
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
    const int bd = blockDim.x;
    for (int i = threadIdx.x; i < np; i += 4 * bd) {
        const double a = partials[i];
        const double b = i + bd < np ? partials[i + bd] : 0.0;
        const double c = i + 2 * bd < np ? partials[i + 2 * bd] : 0.0;
        const double d = i + 3 * bd < np ? partials[i + 3 * bd] : 0.0;
        m0 = fmax(m0, a); m1 = fmax(m1, b); m2 = fmax(m2, c); m3 = fmax(m3, d);
    }
    const double mx = fmax(fmax(m0, m1), fmax(m2, m3));
    sh[threadIdx.x] = mx;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) scalars[slot] = sh[0];
}

// Chebyshev first step: d = c * dinv * r ; x (+)= d
template <bool ZERO_GUESS>
__global__ void __launch_bounds__(kThreads)
    k_cheb_first(const double *__restrict__ r, const double *__restrict__ dinv, double c, double *__restrict__ d,
                 double *__restrict__ x, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double di = c * dinv[i] * r[i];
        d[i] = di;
        x[i] = ZERO_GUESS ? di : x[i] + di;
    }
}

// Chebyshev step k>=2: rout = rin - q ; d = c1 d + c2 dinv rout ; x += d
__global__ void __launch_bounds__(kThreads)
    k_cheb_step(const double *__restrict__ rin, const double *__restrict__ q, const double *__restrict__ dinv, double c1,
                double c2, double *__restrict__ rout, double *__restrict__ d, double *__restrict__ x, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double ri = rin[i] - q[i];
        rout[i] = ri;
        const double di = c1 * d[i] + c2 * dinv[i] * ri;
        d[i] = di;
        x[i] += di;
    }
}

// one CTA: dense inverse of a small CSR matrix by Gauss-Jordan with partial pivoting.  BAND: 1024 threads, each step
// updates only the rows with a nonzero multiplier (see below); the pivots and the inverse are the same doubles as the full
// sweep (!BAND, 256 threads), whose pivot search picks the same row at any thread count (ties go to the lower index).
template <bool BAND, int NT = BAND ? 1024 : kThreads>
__global__ void __launch_bounds__(NT)
    k_dense_inverse(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ vals,
                    int n, double *__restrict__ A, double *__restrict__ Inv) {
    __shared__ double fac[kMgDenseMax];
    __shared__ int rows[BAND ? kMgDenseMax : 1];
    __shared__ int piv, nrows;
    __shared__ double rowA[BAND ? kMgDenseMax : 1], rowI[BAND ? kMgDenseMax : 1];   // the normalised pivot row
    const int tid = threadIdx.x;
    for (int idx = tid; idx < n * n; idx += NT) {
        A[idx] = 0.0;
        Inv[idx] = (idx / n == idx % n) ? 1.0 : 0.0;
    }
    __syncthreads();
    for (int i = tid; i < n; i += NT)
        for (int32_t t = rowptr[i]; t < rowptr[i + 1]; ++t) A[i * n + col[t]] = vals[t];
    __syncthreads();
    __shared__ double pvv[NT];
    __shared__ int pvi[NT];
    for (int k = 0; k < n; ++k) {
        // pivot = first row of maximal |A[i][k]|, i >= k: block-wide argmax (ties to the lower index, as a serial scan would)
        {
            double bv = -1.0;
            int best = k;
            for (int i = k + tid; i < n; i += NT) {
                const double v = fabs(A[i * n + k]);
                if (v > bv) { bv = v; best = i; }
            }
            pvv[tid] = bv;
            pvi[tid] = best;
            __syncthreads();
            for (int o = NT / 2; o > 0; o >>= 1) {
                if (tid < o) {
                    const double v2 = pvv[tid + o];
                    const int i2 = pvi[tid + o];
                    if (v2 > pvv[tid] || (v2 == pvv[tid] && i2 < pvi[tid])) { pvv[tid] = v2; pvi[tid] = i2; }
                }
                __syncthreads();
            }
            if (tid == 0) piv = pvi[0];
        }
        __syncthreads();
        const int pr = piv;
        if (pr != k)
            for (int j = tid; j < n; j += NT) {
                double t = A[k * n + j]; A[k * n + j] = A[pr * n + j]; A[pr * n + j] = t;
                t = Inv[k * n + j]; Inv[k * n + j] = Inv[pr * n + j]; Inv[pr * n + j] = t;
            }
        __syncthreads();
        const double pv = 1.0 / A[k * n + k];
        __syncthreads();
        for (int j = tid; j < n; j += NT) {
            const double a = A[k * n + j] * pv, v = Inv[k * n + j] * pv;
            A[k * n + j] = a;
            Inv[k * n + j] = v;
            if (BAND) { rowA[j] = a; rowI[j] = v; }
        }
        if (BAND) {
            // only the rows with a nonzero multiplier change: list them (in any order, their updates are independent) and
            // sweep each one warp-wide, the same update of the same entries as the full sweep below.  On a lattice coarse
            // level that is the band below the pivot plus the filled rows above it, about half the rows.  Columns <= k of
            // A are never read again (every later read of A is in a column > k), so A is updated right of the pivot only;
            // Inv over all n columns.
            if (tid == 0) nrows = 0;
            __syncthreads();
            for (int i = tid; i < n; i += NT) {
                const double f = (i == k) ? 0.0 : A[i * n + k];
                if (f != 0.0) {
                    fac[i] = f;
                    rows[atomicAdd(&nrows, 1)] = i;
                }
            }
            __syncthreads();
            const int warp = tid >> 5, lane = tid & 31, nr = nrows;
            for (int r = warp; r < nr; r += NT / 32) {
                const int i = rows[r];
                const double f = fac[i];
                for (int j = k + 1 + lane; j < n; j += 32) A[i * n + j] -= f * rowA[j];
                for (int j = lane; j < n; j += 32) Inv[i * n + j] -= f * rowI[j];
            }
        } else {
            for (int i = tid; i < n; i += NT) fac[i] = (i == k) ? 0.0 : A[i * n + k];
            __syncthreads();
            for (int idx = tid; idx < n * n; idx += NT) {
                const int i = idx / n, j = idx % n;
                const double f = fac[i];
                if (f != 0.0) {
                    A[idx] -= f * A[k * n + j];
                    Inv[idx] -= f * Inv[k * n + j];
                }
            }
        }
        __syncthreads();
    }
}

// coarsest-level inverse: the row-compacted sweep unless FEMO_NO_BAND_INVERSE asks for the full one
static inline void launch_dense_inverse(const int32_t *rowptr, const int32_t *col, const double *vals, int n, double *A,
                                        double *Inv, cudaStream_t st) {
    if (g_env.no_band_inverse) k_dense_inverse<false><<<1, kThreads, 0, st>>>(rowptr, col, vals, n, A, Inv);
    else k_dense_inverse<true><<<1, 1024, 0, st>>>(rowptr, col, vals, n, A, Inv);
}

// x = Inv * b (tiny system: one warp per row)
__global__ void __launch_bounds__(kThreads) k_dense_apply(const double *__restrict__ Inv, const double *__restrict__ b,
                                                          double *__restrict__ x, int n) {
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (row >= n) return;
    double acc = 0.0;
    for (int j = lane; j < n; j += 32) acc += Inv[row * n + j] * b[j];
    acc = warp_sum(acc);
    if (lane == 0) x[row] = acc;
}

}  // namespace femo

using namespace femo;

// ===========================================================================
// host side
// ===========================================================================

static long long total_launches(const femo_problem *p) {
    long long n = p->launches;
    for (const femo_problem *c : p->mg) n += c->launches;
    return n;
}

// level lv of the hierarchy: 0 is the root problem itself
static inline femo_problem *mg_level(femo_problem *root, int lv) { return lv == 0 ? root : root->mg[lv - 1]; }

// d = c * dinv * b   (first Chebyshev direction from a zero initial guess)
__global__ void __launch_bounds__(kThreads)
    k_cheb_d0(const double *__restrict__ b, const double *__restrict__ dinv, double c, double *__restrict__ d, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        d[i] = c * dinv[i] * b[i];
}

// ---- matrix-free SIMP operator on uniform hexahedral lattices ------------------------------------------------
// y = A x with A = sum_cells rho_c^p K0 (all cells of a level are congruent boxes, so ONE 24x24 unit-modulus element
// matrix serves the level): no matrix traffic at all, only x, the cell moduli and the Dirichlet marks.  One thread
// per node gathers its 8 cells (fixed order => deterministic).  Dirichlet dofs follow the assembled BC'd matrix:
// masked rows are diag * x, masked columns are skipped.  Used for the SpMVs INSIDE the V-cycle only (a
// preconditioner may be any fixed SPD operator); the Krylov recurrence keeps the assembled matrix it was given.
struct HexLat {
    int nx, ny, nzl;   // local cells per direction; nodes (nx+1)(ny+1)(nzl+1), node = (k*(ny+1)+j)*(nx+1)+i
};

__global__ void __launch_bounds__(kThreads) k_pow_cells(const double *__restrict__ rho, double p, double *__restrict__ ec, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) ec[i] = pow(rho[i], p);
}

// CTA = a 32 x 4 x 2 tile of nodes (a warp = 32 consecutive nodes of one lattice row).  The tile's x values plus a
// one-node halo are staged in shared memory with coalesced loads, component-major ([s][node]: conflict-free reads),
// Dirichlet columns zeroed while staging.  K0 travels as a 4.6 KB kernel parameter: with the cell / node loops fully
// unrolled its entries are constant-bank operands of the FMAs (no load instructions at all).
struct HexK0 {
    double k[576];
};
constexpr int kMfX = 32, kMfY = 4, kMfZ = 2;
constexpr int kMfHX = kMfX + 2, kMfHY = kMfY + 2, kMfHZ = kMfZ + 2, kMfHalo = kMfHX * kMfHY * kMfHZ;

template <int EPI>
__global__ void __launch_bounds__(kThreads)
    k_hex_matfree(HexLat L, const __grid_constant__ HexK0 KP, const double *__restrict__ ec, const uint8_t *__restrict__ mask,
                  const double *__restrict__ bcdiag, const double *__restrict__ x, double *__restrict__ y, SpmvEpi E, int tiles_x,
                  int tiles_y) {
    __shared__ double xs[3 * kMfHalo];
    const int sx = L.nx + 1, sy = L.ny + 1, sz = L.nzl + 1;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int i0 = bx * kMfX - 1, j0 = by * kMfY - 1, k0n = bz * kMfZ - 1;      // lattice index of halo node (0,0,0)
    // stage: rows of the halo box are contiguous runs of 3*kMfHX doubles in x
    for (int row = threadIdx.x / 128; row < kMfHY * kMfHZ; row += kThreads / 128) {
        const int hj = row % kMfHY, hk = row / kMfHY;
        const int j = j0 + hj, k = k0n + hk;
        const int t = threadIdx.x % 128;
        if (t < 3 * kMfHX) {
            const int hi = t / 3, s = t % 3, i = i0 + hi;
            double v = 0.0;
            if (i >= 0 && i < sx && j >= 0 && j < sy && k >= 0 && k < sz) {
                const int64_t q = 3 * ((((int64_t)k * sy) + j) * sx + i) + s;
                v = (mask && mask[q]) ? 0.0 : __ldg(x + q);
            }
            xs[s * kMfHalo + (hk * kMfHY + hj) * kMfHX + hi] = v;
        }
    }
    __syncthreads();
    const int li = threadIdx.x % kMfX, lj = (threadIdx.x / kMfX) % kMfY, lk = threadIdx.x / (kMfX * kMfY);
    const int i = bx * kMfX + li, j = by * kMfY + lj, k = bz * kMfZ + lk;
    if (i >= sx || j >= sy || k >= sz) return;
    double acc[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int dk = -1; dk <= 0; ++dk) {
        const int ck = k + dk;
        if (ck < 0 || ck >= L.nzl) continue;
#pragma unroll
        for (int dj = -1; dj <= 0; ++dj) {
            const int cj = j + dj;
            if (cj < 0 || cj >= L.ny) continue;
#pragma unroll
            for (int di = -1; di <= 0; ++di) {
                const int ci = i + di;
                if (ci < 0 || ci >= L.nx) continue;
                const double e = __ldg(ec + ((int64_t)ck * L.ny + cj) * L.nx + ci);
                const int a = (-di) + 2 * (-dj) + 4 * (-dk);              // this node's corner in that cell
                // halo-local index of the cell's node 0: (li+1+di, lj+1+dj, lk+1+dk)
                const int h0 = ((lk + 1 + dk) * kMfHY + (lj + 1 + dj)) * kMfHX + (li + 1 + di);
                double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const int h = h0 + (b & 1) + ((b >> 1) & 1) * kMfHX + (b >> 2) * kMfHX * kMfHY;
                    const double x0 = xs[h], x1 = xs[kMfHalo + h], x2 = xs[2 * kMfHalo + h];
                    const double *Kr = KP.k + (3 * a) * 24 + 3 * b;     // compile-time offsets after unrolling: constant-bank operands
                    s0 += Kr[0] * x0 + Kr[1] * x1 + Kr[2] * x2;
                    s1 += Kr[24] * x0 + Kr[25] * x1 + Kr[26] * x2;
                    s2 += Kr[48] * x0 + Kr[49] * x1 + Kr[50] * x2;
                }
                acc[0] += e * s0;
                acc[1] += e * s1;
                acc[2] += e * s2;
            }
        }
    }
    const int64_t node = (((int64_t)k * sy) + j) * sx + i;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int64_t row = 3 * node + r;
        const double xi = __ldg(x + row);
        const double v = (mask && mask[row]) ? bcdiag[row] * xi : acc[r];
        spmv_row_epilogue<EPI>(E, row, v, xi, y);
    }
}

static inline bool hex_matfree_ready(const femo_problem *L) {
    return L->mgl.ec && L->mgl.k0 && L->h_k0.size() == 576 && L->family == FEMO_FAMILY_SIMP_HEX8;
}

static int launch_hex_matfree(femo_problem *L, int kind, const double *x, double *y, const SpmvEpi &E) {
    int rc = halo_nodes(L, const_cast<double *>(x));
    if (rc) return rc;
    const HexLat H{L->mesh.n[0], L->mesh.n[1], L->mesh.n[2]};
    const uint8_t *mk = L->has_bc ? L->d_bc_mark : nullptr;
    const int tx = (H.nx + 1 + kMfX - 1) / kMfX, ty = (H.ny + 1 + kMfY - 1) / kMfY, tz = (H.nzl + 1 + kMfZ - 1) / kMfZ;
    const int g = tx * ty * tz;
    HexK0 KP;
    memcpy(KP.k, L->h_k0.data(), sizeof(KP.k));
    if (kind == EPI_PLAIN) k_hex_matfree<EPI_PLAIN><<<g, kThreads, 0, L->stream>>>(H, KP, L->mgl.ec, mk, L->d_bc_diag, x, y, E, tx, ty);
    else if (kind == EPI_CHEB0) k_hex_matfree<EPI_CHEB0><<<g, kThreads, 0, L->stream>>>(H, KP, L->mgl.ec, mk, L->d_bc_diag, x, y, E, tx, ty);
    else k_hex_matfree<EPI_CHEBK><<<g, kThreads, 0, L->stream>>>(H, KP, L->mgl.ec, mk, L->d_bc_diag, x, y, E, tx, ty);
    L->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

__global__ void __launch_bounds__(kThreads) k_to_f32(const double *__restrict__ a, float *__restrict__ o, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) o[i] = (float)a[i];
}

// ---- DIA (stencil) levels ------------------------------------------------------------------------------------
static inline bool dia_ready(const femo_problem *L) { return L->mgl.dia_valid; }

// The representation of a level's operator that the V-cycle streams: at fp32 the matrix-free hexahedral operator, else
// the DIA planes, else the fp32 CSR copy; fp64 CSR otherwise.  Decided per call, not stored: the Chebyshev
// preconditioner (precond 1) smooths the root at fp64 without a multigrid set-up.  The first two never compete: DIA
// planes exist on triangle lattices only, the matrix-free operator on hexahedral ones.
enum class LevelOp { MATFREE, DIA, CSR32, CSR64 };
static inline LevelOp level_op(const femo_problem *L, bool fp32) {
    if (fp32 && hex_matfree_ready(L)) return LevelOp::MATFREE;
    if (fp32 && dia_ready(L)) return LevelOp::DIA;
    if (fp32 && L->mgl.vals32) return LevelOp::CSR32;
    return LevelOp::CSR64;
}

// column offsets of a scalar vertex space on a right-diagonal triangle lattice: the node itself, its x / y
// neighbours and the two ends of the cell diagonals
static inline bool dia_offsets(const femo_problem *L, DiaMat &A) {
    if (g_env.no_dia) return false;
    if (!(L->mesh.lattice && L->mesh.kind == MESH_TRI && L->state.element == EL_VERTEX && L->state.block == 1)) return false;
    const int w = L->mesh.n[0] + 1;
    const int off[7] = {-w - 1, -w, -1, 0, 1, w, w + 1};
    A.nd = 7;
    A.sdiag = 3;
    for (int s = 0; s < 7; ++s) A.off[s] = off[s];
    A.n = L->state.ndofs;
    A.np = (A.n + 31) & ~(int64_t)31;
    return true;
}
// the level's Jacobian can be assembled node-centrically straight into its DIA planes (lattice_jacobian with_dia)
static inline bool lattice_dia_direct(const femo_problem *L) {
    DiaMat tmp;
    return L->lattice_fast && L->mgl.vals32 && dia_offsets(L, tmp) && !g_env.no_lattice_asm;
}
// floats reserved for the fp32 operator copy of a level: the CSR copy or the DIA planes, whichever is larger
static inline size_t fp32_copy_len(const femo_problem *L) {
    DiaMat A;
    size_t n = (size_t)L->pat[0].nnz;
    if (dia_offsets(L, A)) n = std::max<size_t>(n, (size_t)(A.nd + 1) * (size_t)A.np);   // + the dinv plane
    return n;
}

// re-layout the level's assembled (BC'd) values as DIA planes in the fp32 buffer; vperm: the level's values are
// M.vals[vperm[t]] (the transpose of M.vals through the square pattern's t_perm)
static int dia_convert(femo_problem *L, const int32_t *vperm = nullptr) {
    femo_mg_level &M = L->mgl;
    DiaMat A;
    if (!dia_offsets(L, A) || !M.vals32) return FEMO_OK;
    const DevPattern &D = L->dpat[0];
    A.v = M.vals32;
    // one pass: planes, dinv and the Gershgorin partial maxima (needs <= kMaxPartials CTAs: finalised in chunks below)
    const int g = grid_for(A.n);
    double *part = L->d_scratch ? L->d_scratch : L->d_partials;      // per-CTA maxima: the element scratch is free here
    if ((size_t)g > L->scratch_len) return set_err(FEMO_ESTATE, "DIA conversion: scratch too small for the partial maxima");
    if (vperm)
        k_csr_to_dia<7, true><<<g, kThreads, 0, L->stream>>>(D.rowptr, D.col, M.vals, A, M.vals32,
                                                             reinterpret_cast<int *>(L->d_scalars + S_FLAG), M.dinv,
                                                             L->own_off, L->own_off + L->own_n, part, M.dia64, vperm);
    else
        k_csr_to_dia<7><<<g, kThreads, 0, L->stream>>>(D.rowptr, D.col, M.vals, A, M.vals32,
                                                       reinterpret_cast<int *>(L->d_scalars + S_FLAG), M.dinv, L->own_off,
                                                       L->own_off + L->own_n, part, M.dia64);
    M.dia64_valid = M.dia64 != nullptr;
    k_max_finalize<<<1, kThreads, 0, L->stream>>>(part, g, L->d_scalars, S_TMP2);
    L->launches += 2;
    FEMO_CHECK_LAUNCH();
    M.dia = A;
    M.dia_valid = true;
    // the fused pre-smoother scales NEIGHBOUR entries by their 1/a_jj: ghost rows need the owner's scaling
    return halo_nodes_f32(L, M.vals32 + (size_t)A.nd * A.np);
}

static void dia_dispatch(int mode, const DiaMat &A, const double *x, double *y, const DiaEpi &E, int nrows, cudaStream_t st) {
    const int g = grid_for(nrows);
    switch (mode) {
        case DIA_PLAIN: k_dia_apply<DIA_PLAIN, 7><<<g, kThreads, 0, st>>>(A, x, y, E); break;
        case DIA_CHEB0: k_dia_apply<DIA_CHEB0, 7><<<g, kThreads, 0, st>>>(A, x, y, E); break;
        case DIA_CHEBK: k_dia_apply<DIA_CHEBK, 7><<<g, kThreads, 0, st>>>(A, x, y, E); break;
        default: k_dia_apply<DIA_PRE2, 7><<<g, kThreads, 0, st>>>(A, x, y, E); break;
    }
}

static int launch_dia(femo_problem *L, int mode, const double *x, double *y, const DiaEpi &E) {
    const DiaMat &A = L->mgl.dia;
    double *in = const_cast<double *>(mode == DIA_PRE2 ? E.b : x);
    int rc;
    RowSplit R;
    if (overlap_begin(L, in, R, &rc)) {
        // slab level: boundary rows behind the exchange on the side stream, interior rows at once on the main stream
        DiaEpi Eb = E, Ei = E;
        Eb.a0 = R.b0; Eb.n0 = R.nb0; Eb.a1 = R.b1; Eb.n1 = R.nb1;
        Ei.a0 = R.i0; Ei.n0 = R.ni; Ei.a1 = 0; Ei.n1 = 0;
        dia_dispatch(mode, A, x, y, Eb, R.nb0 + R.nb1, L->stream2);
        dia_dispatch(mode, A, x, y, Ei, R.ni, L->stream);
        L->launches += 2;
        L->dia_count[mode & 3]++;
        FEMO_CHECK_LAUNCH();
        return overlap_end(L);
    }
    if (rc) return rc;
    if ((rc = halo_nodes(L, in))) return rc;
    dia_dispatch(mode, A, x, y, E, (int)A.n, L->stream);
    L->launches++;
    L->dia_count[mode & 3]++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// y = A x (or bsub - A x) with the level's fp64 planes; DOT: fused partial sums of x.y over the owned rows
template <bool DOT>
static int launch_dia64(femo_problem *L, const double *x, double *y, const double *bsub, int *np_out) {
    const DiaMat &A = L->mgl.dia;
    const int64_t cap = std::min<int64_t>((int64_t)L->num_sms * 8, kMaxPartials - 64);
    int rc;
    RowSplit R;
    if (overlap_begin(L, const_cast<double *>(x), R, &rc)) {
        // interior partial sums first, the boundary launch's behind them: fixed layout => deterministic reduction
        const int gi = (int)std::max<int64_t>(1, std::min<int64_t>(grid_for(R.ni), cap));
        const int gb = (int)std::max<int64_t>(1, std::min<int64_t>(grid_for(R.nb0 + R.nb1), 64));
        k_dia_spmv64<DOT, 7><<<gb, kThreads, 0, L->stream2>>>(L->mgl.dia64, A, x, y, bsub, L->own_off, L->own_off + L->own_n,
                                                              L->d_partials + gi, R.b0, R.nb0, R.b1, R.nb1);
        k_dia_spmv64<DOT, 7><<<gi, kThreads, 0, L->stream>>>(L->mgl.dia64, A, x, y, bsub, L->own_off, L->own_off + L->own_n,
                                                             L->d_partials, R.i0, R.ni, 0, 0);
        L->launches += 2;
        L->dia64_count[DOT ? 0 : 1]++;
        if (np_out) *np_out = gi + gb;
        FEMO_CHECK_LAUNCH();
        return overlap_end(L);
    }
    if (rc) return rc;
    if ((rc = halo_nodes(L, const_cast<double *>(x)))) return rc;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(grid_for(A.n), cap));
    k_dia_spmv64<DOT, 7><<<grid, kThreads, 0, L->stream>>>(L->mgl.dia64, A, x, y, bsub, L->own_off, L->own_off + L->own_n,
                                                           L->d_partials, 0, -1, 0, 0);
    L->launches++;
    L->dia64_count[DOT ? 0 : 1]++;
    if (np_out) *np_out = grid;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// one application of the level operator `op` with the row epilogue `kind`: EPI_PLAIN y = b - A x (b = E.b), or the
// Chebyshev steps EPI_CHEB0 / EPI_CHEBK, whose outputs E names
static int level_apply(femo_problem *L, LevelOp op, int kind, const double *x, double *y, const SpmvEpi &E) {
    femo_mg_level &M = L->mgl;
    const DevPattern &D = L->dpat[0];
    switch (op) {
        case LevelOp::MATFREE: return launch_hex_matfree(L, kind, x, y, E);
        case LevelOp::DIA: {
            DiaEpi De;
            De.b = E.b; De.rin = E.rin; De.rout = E.rout; De.dout = E.dout; De.xacc = E.xacc;
            De.c1 = E.c1; De.c2 = E.c2; De.xmode = E.xmode;
            return launch_dia(L, kind == EPI_PLAIN ? DIA_PLAIN : kind == EPI_CHEB0 ? DIA_CHEB0 : DIA_CHEBK, x, y, De);
        }
        case LevelOp::CSR32:
            if (kind == EPI_PLAIN) return launch_spmv<false>(L, D.rb, D.nrb, D.rowptr, D.col, M.vals32, x, y, E.b, nullptr);
            return launch_spmv_cheb(L, kind, M.vals32, x, E);
        default:
            if (kind == EPI_PLAIN) return launch_spmv<false>(L, D.rb, D.nrb, D.rowptr, D.col, M.vals, x, y, E.b, nullptr);
            return launch_spmv_cheb(L, kind, M.vals, x, E);
    }
}

// degree and interval [lmax / ratio, lmax] of a Chebyshev-Jacobi smoother
struct ChebParams {
    int degree = 2;
    double ratio = 4.0;
};
struct MgParams : ChebParams {
    bool fp32 = true;      // V-cycle SpMVs stream fp32 copies of the level matrices (vectors stay fp64)
};

// Chebyshev polynomial of the Jacobi-scaled operator on [lmax / ratio, lmax]: d_1 = c0 D^-1 r_0, then every further step
// d_k = c1 d_{k-1} + c2 D^-1 r_{k-1} with rho_1 = 1 / sigma, rho_k = 1 / (2 sigma - rho_{k-1}).  Every smoother path
// (cheb_smooth, the fused PRE2 kernel, the level sweeps, the cooperative coarse V-cycle) takes its coefficients from
// here, so each is the same double.
struct ChebPoly {
    double theta, delta, sigma, rho, c0, c1 = 0.0, c2 = 0.0;
    ChebPoly(double lmax, double ratio) {
        const double lmin = lmax / ratio;
        theta = 0.5 * (lmax + lmin);
        delta = 0.5 * (lmax - lmin);
        sigma = theta / delta;
        rho = 1.0 / sigma;
        c0 = 1.0 / theta;
    }
    void next() {          // c1, c2 of the next step
        const double rho_new = 1.0 / (2.0 * sigma - rho);
        c1 = rho_new * rho;
        c2 = 2.0 * rho_new / delta;
        rho = rho_new;
    }
};

// work vectors of a smoothed level (Jacobi scaling, residual, two directions), its rows and its Gershgorin bound
struct ChebWork {
    const double *dinv;
    double *r, *d, *q;
    int64_t n;
    double lmax;
};

// Chebyshev-Jacobi smoother of degree `deg`: x ~ A^-1 b.  Every step after the first is ONE operator application,
// apply(kind, x, E) with kind EPI_CHEB0 / EPI_CHEBK, that carries the residual / direction / solution updates in its row
// epilogue.  Kernels run on p's stream and count on p.  drop_last: the last step stores no residual / direction.
template <class Apply>
static int cheb_smooth(femo_problem *p, const ChebWork &W, const double *b, double *x, bool zero_guess, int deg, double ratio,
                       bool drop_last, const Apply &apply) {
    const int64_t n = W.n;
    cudaStream_t st = p->stream;
    const int g = red_grid(p, n);
    ChebPoly P(W.lmax, ratio);
    int rc;
    double *dcur = W.d, *dnext = W.q;
    const double *rin;
    int xmode;
    if (zero_guess) {
        if (deg <= 1) {
            k_cheb_first<true><<<g, kThreads, 0, st>>>(b, W.dinv, P.c0, dcur, x, n);
            p->launches++;
            FEMO_CHECK_LAUNCH();
            return FEMO_OK;
        }
        k_cheb_d0<<<g, kThreads, 0, st>>>(b, W.dinv, P.c0, dcur, n);
        p->launches++;
        rin = b;
        xmode = 2;                 // x = d0 + d1
    } else {
        SpmvEpi E;                 // r = b - A x ; d0 = dinv r / theta
        E.b = b; E.dinv = W.dinv; E.rout = W.r; E.dout = dcur; E.c1 = P.c0;
        if ((rc = apply(EPI_CHEB0, x, E))) return rc;
        if (deg <= 1) {
            k_axpy<<<g, kThreads, 0, st>>>(1.0, dcur, x, n);
            p->launches++;
            FEMO_CHECK_LAUNCH();
            return FEMO_OK;
        }
        rin = W.r;
        xmode = 1;                 // x += d0 + d1
    }
    for (int k = 2; k <= deg; ++k) {
        P.next();
        SpmvEpi E;
        E.dinv = W.dinv; E.rin = rin; E.rout = W.r; E.dout = dnext; E.xacc = x;
        E.c1 = P.c1; E.c2 = P.c2; E.xmode = xmode;
        if (drop_last && k == deg) E.rout = E.dout = nullptr;      // nobody reads the last residual / direction
        if ((rc = apply(EPI_CHEBK, dcur, E))) return rc;
        std::swap(dcur, dnext);
        rin = W.r;
        xmode = 0;
    }
    return FEMO_OK;
}

// the smoother of a geometric level; DIA levels add two shortcuts of k_dia_apply: the zero-guess degree-2 smoother as
// one kernel, and no residual / direction stored by the last step (the kernel skips null outputs)
static int mg_smooth(femo_problem *L, const double *b, double *x, bool zero_guess, int deg, double ratio, bool fp32) {
    femo_mg_level &M = L->mgl;
    const LevelOp op = level_op(L, fp32);
    if (zero_guess && deg == 2 && op == LevelOp::DIA) {     // d0, the operator and both updates in one kernel
        ChebPoly P(M.lmax, ratio);
        P.next();
        DiaEpi E;
        E.b = b; E.c0 = P.c0; E.c1 = P.c1; E.c2 = P.c2;
        return launch_dia(L, DIA_PRE2, nullptr, x, E);
    }
    return cheb_smooth(L, ChebWork{M.dinv, M.r, M.d, M.q, L->state.ndofs, M.lmax}, b, x, zero_guess, deg, ratio,
                       op == LevelOp::DIA, [&](int kind, const double *xin, const SpmvEpi &E) {
                           return level_apply(L, op, kind, xin, nullptr, E);
                       });
}

static inline LatD latd_of(const femo_problem *p) {
    return LatD{p->mesh.n[0], p->mesh.n[1] + 1, p->slab.active ? p->slab.crow0 : 0};
}
// global cell rows of a level (slab: of the partitioned lattice)
static inline int global_rows(const femo_problem *p) { return p->slab.active ? p->slab.gny : p->mesh.n[1]; }
static inline LatD3 latd3_of(const femo_problem *p) {
    return LatD3{p->mesh.n[0], p->mesh.n[1], p->mesh.n[2] + 1, p->slab.active ? p->slab.crow0 : 0};
}
// dofs in one slab row (a lattice row in 2-D, a z-plane of nodes for hexahedra)
static inline size_t slab_row_len(const femo_problem *p) {
    return (size_t)(p->mesh.n[0] + 1) * (p->mesh.kind == MESH_HEX ? (size_t)(p->mesh.n[1] + 1) : 1) * p->state.block;
}
static inline int slab_axis_cells(const femo_problem *p) { return p->mesh.kind == MESH_HEX ? p->mesh.n[2] : p->mesh.n[1]; }
static inline bool nested_pair(const femo_problem *F, const femo_problem *C) {
    if (F->mesh.kind == MESH_HEX && F->state.element == EL_VERTEX) {
        const int gf = F->slab.active ? F->slab.gny : F->mesh.n[2], gc = C->slab.active ? C->slab.gny : C->mesh.n[2];
        return F->mesh.n[0] == 2 * C->mesh.n[0] && F->mesh.n[1] == 2 * C->mesh.n[1] && gf == 2 * gc;
    }
    if (F->mesh.kind != MESH_TRI || F->state.block != 1) return false;   // integer-only kernels: scalar P1
    return F->mesh.n[0] == 2 * C->mesh.n[0] && global_rows(F) == 2 * global_rows(C);
}

static int mg_restrict(femo_problem *L, femo_problem *C, double *rf, double *rc_);
static int mg_prolong_add(femo_problem *L, femo_problem *C, double *xc, double *xf);
static int mgfused_vcycle(femo_problem *root, int lv, const double *b, double *x, const MgParams &mp, bool *done);
static int mgsweep_vcycle(femo_problem *root, int lv, const double *b, double *x, const MgParams &mp, bool *done);

// one V-cycle: level lv solves A x = b approximately from a zero initial guess.  Levels <= FEMO_MGFUSED_MAX_ROWS run
// as one cooperative kernel (mgfused.cuh); single-GPU DIA levels above that range with a 2:1 nested coarse level run
// their visit as two stencil sweeps (mgsweep.cuh); every other level takes the per-kernel path below.
static int mg_vcycle(femo_problem *root, int lv, const double *b, double *x, const MgParams &mp) {
    femo_problem *L = mg_level(root, lv);
    const int nlev = (int)root->mg.size() + 1;
    femo_mg_level &M = L->mgl;
    const int64_t n = L->state.ndofs;
    cudaStream_t st = L->stream;
    int rc;
    if (lv == nlev - 1) {
        k_dense_apply<<<(int)((n * 32 + kThreads - 1) / kThreads), kThreads, 0, st>>>(M.dense, b, x, (int)n);
        L->launches++;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    {   // coarse levels: the whole sub-V-cycle in one cooperative kernel (mgfused.cuh)
        bool done = false;
        if ((rc = mgfused_vcycle(root, lv, b, x, mp, &done))) return rc;
        if (done) return FEMO_OK;
    }
    {   // large DIA levels: the whole visit in two stencil sweeps around the coarse correction (mgsweep.cuh)
        bool done = false;
        if ((rc = mgsweep_vcycle(root, lv, b, x, mp, &done))) return rc;
        if (done) return FEMO_OK;
    }
    femo_problem *C = root->mg[lv];
    femo_mg_level &MC = C->mgl;
    if ((rc = mg_smooth(L, b, x, true, mp.degree, mp.ratio, mp.fp32))) return rc;
    // r = b - A x ; restrict
    SpmvEpi E;
    E.b = b;
    if ((rc = level_apply(L, level_op(L, mp.fp32), EPI_PLAIN, x, M.r, E))) return rc;
    if ((rc = mg_restrict(L, C, M.r, MC.b))) return rc;
    if ((rc = mg_vcycle(root, lv + 1, MC.b, MC.x, mp))) return rc;
    if ((rc = mg_prolong_add(L, C, MC.x, x))) return rc;
    // x had fresh ghost rows for the residual SpMV and the nested prolongation corrected them from the (exchanged)
    // coarse ghost rows: the post-smoother's first SpMV needs no halo exchange
    L->skip_next_halo = L->slab.active && nested_pair(L, C);
    return mg_smooth(L, b, x, false, mp.degree, mp.ratio, mp.fp32);
}

// transfers between level lv (fine) and lv+1 (coarse) of the hierarchy, shared by the V-cycle and the
// full-multigrid start: rc = P^T rf (replicated coarse levels are gathered), xf (+)= P xc
static int mg_restrict(femo_problem *L, femo_problem *C, double *rf, double *rc_) {
    const int64_t nc = C->state.ndofs;
    const uint8_t *mf = L->has_bc ? L->d_bc_mark : nullptr, *mc = C->has_bc ? C->d_bc_mark : nullptr;
    cudaStream_t st = L->stream;
    int rc;
    if (L->state.element == EL_P2) {                               // p-multigrid: P2 -> P1 on the same mesh
        k_p2_to_p1_restrict<<<grid_for(nc), kThreads, 0, st>>>(L->d_vptr, L->d_vedge, L->mesh.nverts, rf, rc_, mf, mc);
        L->launches++;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    if (nested_pair(L, C)) {
        if ((rc = halo_nodes(L, rf))) return rc;                  // coarse owned rows read the fine ghost row below
        if (L->mesh.kind == MESH_HEX)
            k_restrict_nested3<<<grid_for(nc), kThreads, 0, st>>>(latd3_of(L), latd3_of(C), L->state.block, rf, rc_, mf, mc);
        else
            k_restrict_nested<<<grid_for(nc), kThreads, 0, st>>>(latd_of(L), latd_of(C), rf, rc_, mf, mc);
        L->launches++;
        if (L->slab.active && !C->slab.active)                     // distributed -> replicated level
            if ((rc = gather_rows(L, rc_, slab_row_len(C), slab_axis_cells(C)))) return rc;
    } else {
        if (L->slab.active) return set_err(FEMO_ESTATE, "distributed multigrid levels must be 2:1 nested");
        if (L->mesh.kind == MESH_HEX)
            k_lattice3_restrict<<<grid_for(nc), kThreads, 0, st>>>(lat3_of(L->mesh), lat3_of(C->mesh), L->state.block, rf, rc_, mf, mc);
        else
            k_lattice_restrict<<<grid_for(nc), kThreads, 0, st>>>(Lattice{L->mesh.n[0], L->mesh.n[1]}, Lattice{C->mesh.n[0], C->mesh.n[1]}, L->state.block, L->mesh.kind == MESH_QUAD, rf, rc_, mf, mc);
        L->launches++;
    }
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

static int mg_prolong_add(femo_problem *L, femo_problem *C, double *xc, double *xf) {
    const int64_t n = L->state.ndofs;
    const uint8_t *mf = L->has_bc ? L->d_bc_mark : nullptr;
    cudaStream_t st = L->stream;
    int rc;
    if (L->state.element == EL_P2) {
        k_p1_to_p2<true><<<grid_for(n), kThreads, 0, st>>>(L->d_edge_verts, L->mesh.nverts, L->mesh.nedges, xc, xf, mf);
        L->launches++;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    if (nested_pair(L, C)) {
        if ((rc = halo_nodes(C, xc))) return rc;                   // fine owned rows read the coarse ghost row above
        if (L->mesh.kind == MESH_HEX)
            k_prolong_nested3<<<grid_for(n), kThreads, 0, st>>>(latd3_of(L), latd3_of(C), L->state.block, xc, xf, mf);
        else
            k_prolong_nested<<<grid_for(n), kThreads, 0, st>>>(latd_of(L), latd_of(C), xc, xf, mf);
    } else if (L->mesh.kind == MESH_HEX) {
        k_lattice3_interp<true><<<grid_for(n), kThreads, 0, st>>>(lat3_of(C->mesh), lat3_of(L->mesh), L->state.block, xc, xf, mf);
    } else {
        k_lattice_interp<true><<<grid_for(n), kThreads, 0, st>>>(Lattice{C->mesh.n[0], C->mesh.n[1]}, Lattice{L->mesh.n[0], L->mesh.n[1]}, L->state.block, L->mesh.kind == MESH_QUAD, xc, xf, mf);
    }
    L->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// Full-multigrid start (nested iteration): x0 ~ A^-1 b to discretisation accuracy for about 1.5 V-cycles
// of work.  Coarsest level solved exactly; each finer level prolongs the coarser iterate and corrects
// it with one V-cycle on its residual.
static int mg_fmg(femo_problem *root, const double *b, double *x, const MgParams &mp) {
    const int nlev = (int)root->mg.size() + 1;
    int rc;
    // right-hand sides of all levels
    for (int lv = 0; lv + 1 < nlev; ++lv) {
        femo_problem *L = mg_level(root, lv), *C = mg_level(root, lv + 1);
        double *rf = (lv == 0) ? const_cast<double *>(b) : L->mgl.fb;
        if ((rc = mg_restrict(L, C, rf, C->mgl.fb))) return rc;
    }
    for (int lv = nlev - 1; lv >= 0; --lv) {
        femo_problem *L = mg_level(root, lv);
        femo_mg_level &M = L->mgl;
        const int64_t n = L->state.ndofs;
        cudaStream_t st = L->stream;
        const double *bl = (lv == 0) ? b : M.fb;
        double *xl = (lv == 0) ? x : M.fx;
        if (lv == nlev - 1) {
            k_dense_apply<<<(int)((n * 32 + kThreads - 1) / kThreads), kThreads, 0, st>>>(M.dense, bl, xl, (int)n);
            L->launches++;
            continue;
        }
        femo_problem *C = mg_level(root, lv + 1);
        FEMO_CUDA(cudaMemsetAsync(xl, 0, sizeof(double) * n, st));
        if ((rc = mg_prolong_add(L, C, C->mgl.fx, xl))) return rc;
        // residual of the prolonged iterate into M.b (free at this level), V-cycle correction into M.x
        double *rl = (lv == 0) ? root->kr_r : M.b, *el = (lv == 0) ? root->kr_z : M.x;
        // residual of the nested iterate: fp64 planes on the fine level, the V-cycle's fp32 planes below, fp64 CSR on
        // every other level, matrix-free and CSR32 ones included (the full-multigrid iterate is only the Krylov
        // method's initial guess)
        const bool dia = level_op(L, mp.fp32) == LevelOp::DIA;
        if (dia && M.dia64_valid) rc = launch_dia64<false>(L, xl, rl, bl, nullptr);
        else {
            SpmvEpi E;
            E.b = bl;
            rc = level_apply(L, dia && lv > 0 ? LevelOp::DIA : LevelOp::CSR64, EPI_PLAIN, xl, rl, E);
        }
        if (rc) return rc;
        if ((rc = mg_vcycle(root, lv, rl, el, mp))) return rc;
        k_axpy<<<red_grid(L, n), kThreads, 0, st>>>(1.0, el, xl, n);
        L->launches++;
        FEMO_CHECK_LAUNCH();
    }
    return FEMO_OK;
}

__global__ void __launch_bounds__(kThreads) k_u8_to_f64(const uint8_t *__restrict__ a, double *__restrict__ b, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) b[i] = a[i] ? 1.0 : 0.0;
}

// Dirichlet marks of the first replicated level: injected from the finest distributed marks each rank
// owns, gathered over the ranks, then installed (and propagated to the coarser replicated levels) on the host
static int sync_replicated_bc(femo_problem *root) {
    size_t g = 0;
    while (g < root->mg.size() && !root->mg[g]->replicated) ++g;
    root->mg_bc_dirty = false;
    if (g == root->mg.size()) return FEMO_OK;
    femo_problem *F = mg_level(root, (int)g);
    femo_problem *C = root->mg[g];
    const int64_t nf = F->state.ndofs, nc = C->state.ndofs;
    cudaStream_t st = root->stream;
    int rc;
    double *tf = F->mgl.r, *tc = C->mgl.x;
    k_u8_to_f64<<<grid_for(nf), kThreads, 0, st>>>(F->d_bc_mark, tf, nf);
    if (F->mesh.kind == MESH_HEX)
        k_inject_nested3<<<grid_for(nc), kThreads, 0, st>>>(latd3_of(F), latd3_of(C), F->state.block, tf, tc);
    else
        k_inject_nested<<<grid_for(nc), kThreads, 0, st>>>(latd_of(F), latd_of(C), tf, tc);
    root->launches += 2;
    FEMO_CHECK_LAUNCH();
    if ((rc = gather_rows(F, tc, slab_row_len(C), slab_axis_cells(C)))) return rc;
    std::vector<double> h(nc);
    FEMO_CUDA(cudaMemcpyAsync(h.data(), tc, sizeof(double) * nc, cudaMemcpyDeviceToHost, st));
    FEMO_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> list;
    for (int64_t i = 0; i < nc; ++i)
        if (h[i] > 0.5) list.push_back((int32_t)i);
    int32_t ptr[2] = {0, (int32_t)list.size()};
    if ((rc = set_bc_impl(C, list.data(), ptr, list.empty() ? 0 : 1, nullptr))) return rc;
    return propagate_bc(root, (int)g + 1);
}

// A CG solve with the fp32 geometric multigrid reads the fine level's CSR values only through its DIA conversion when
// the fine level converts (mg_setup's DIA branch: lattice P1, fp32 and fp64 planes, not the coarsest level): the V-cycle
// streams the fp32 planes, the recurrence and the full-multigrid residual the fp64 planes.  Then a transposed solve can
// convert through the pattern's t_perm instead of permuting every value first.
static bool level0_dia_only(const femo_problem *p, const femo_krylov_opts &o) {
    DiaMat A;
    return o.method == 0 && o.precond == 2 && o.mg_precision == 0 && !p->mg.empty() && p->dpat[0].t_perm &&
           !hex_matfree_ready(p) && p->mgl.vals32 && p->mgl.dia64 && dia_offsets(p, A);
}

// (re)build the hierarchy for the matrix `vals` of the root at the root's current state
// level0_dia: the caller has just assembled `vals` with lattice_jacobian(..., with_dia = true): the fine level's DIA
// planes, dinv and Gershgorin maximum are already in place
// vperm: the fine level's matrix is vals[vperm[t]] (see level0_dia_only); only its DIA conversion may read `vals`
static int mg_setup(femo_problem *root, const double *vals, bool fp32 = true, bool level0_dia = false,
                    const int32_t *vperm = nullptr) {
    if (root->mg.empty()) return set_err(FEMO_ESTATE, "multigrid requested but femo_problem_enable_multigrid was not called before upload");
    if (vperm && level0_dia) return set_err(FEMO_ESTATE, "multigrid setup: gathered values cannot come with DIA planes");
    const int nlev = (int)root->mg.size() + 1;
    int rc;
    if (root->mg_bc_dirty && (rc = sync_replicated_bc(root))) return rc;
    if (root->coef[0] && (rc = halo_nodes(root, const_cast<double *>(root->coef[0])))) return rc;
    // Every level's Gershgorin bound and DIA error flag (its S_TMP2 .. S_FLAG) is copied into the root's S_MG slots on the
    // stream, and all of them come to the host in one read once every level is enqueued.  No level's set-up reads a
    // host-side lmax: only the smoothers and the fused coarse program use it, and they run after the set-up.
    constexpr int kSlots = S_FLAG - S_TMP2 + 1, kBatch = (S_COUNT - S_MG) / kSlots;
    femo_problem *pend[kBatch];
    int npend = 0;
    auto flush = [&]() -> int {
        if (!npend) return FEMO_OK;
        double lm[kBatch * kSlots];
        int rc2 = read_scalars(root, S_MG, npend * kSlots, lm);
        if (rc2) return rc2;
        for (int j = 0; j < npend; ++j) {
            pend[j]->mgl.lmax = lm[j * kSlots];
            if (lm[j * kSlots + S_FLAG - S_TMP2] != 0.0)
                return set_err(FEMO_ESTATE, "DIA conversion met a column offset outside the lattice stencil");
        }
        npend = 0;
        return FEMO_OK;
    };
    for (int lv = 0; lv < nlev; ++lv) {
        femo_problem *L = mg_level(root, lv);
        femo_mg_level &M = L->mgl;
        cudaStream_t st = L->stream;
        const int64_t n = L->state.ndofs;
        bool direct = lv == 0 && level0_dia && fp32 && dia_ready(L);     // DIA planes written by the assembly itself
        if (lv == 0) {
            M.vals = const_cast<double *>(vals);
        } else {
            femo_problem *F = mg_level(root, lv - 1);
            const double *uf = (lv == 1) ? root->coef[0] : F->mgl.u;
            if (!uf) return set_err(FEMO_ESTATE, "multigrid setup: state coefficient not set");
            if (F->state.element == EL_P2) {                      // vertex values of the P2 state
                FEMO_CUDA(cudaMemcpyAsync(M.u, uf, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, st));
            } else if (nested_pair(F, L)) {
                if (L->mesh.kind == MESH_HEX)
                    k_inject_nested3<<<grid_for(n), kThreads, 0, st>>>(latd3_of(F), latd3_of(L), L->state.block, uf, M.u);
                else
                    k_inject_nested<<<grid_for(n), kThreads, 0, st>>>(latd_of(F), latd_of(L), uf, M.u);
                L->launches++;
                if (L->slab.active) {
                    if ((rc = halo_nodes(L, M.u))) return rc;      // the ghost row below has no local fine parent
                } else if (F->slab.active) {
                    if ((rc = gather_rows(F, M.u, slab_row_len(L), slab_axis_cells(L)))) return rc;
                }
            } else {
                if (F->slab.active) return set_err(FEMO_ESTATE, "distributed multigrid levels must be 2:1 nested");
                if (L->mesh.kind == MESH_HEX)
                    k_lattice3_interp<false><<<grid_for(n), kThreads, 0, st>>>(lat3_of(F->mesh), lat3_of(L->mesh), L->state.block, uf, M.u, nullptr);
                else
                    k_lattice_interp<false><<<grid_for(n), kThreads, 0, st>>>(Lattice{F->mesh.n[0], F->mesh.n[1]}, Lattice{L->mesh.n[0], L->mesh.n[1]}, L->state.block, L->mesh.kind == MESH_QUAD, uf, M.u, nullptr);
                L->launches++;
            }
            L->coef[0] = M.u;
            L->coefn[0] = n;
            if (L->family == FEMO_FAMILY_SIMP_HEX8) {
                const double *mf_ = (lv == 1) ? root->coef[1] : F->mgl.m;
                if (!mf_) return set_err(FEMO_ESTATE, "multigrid setup: density coefficient not set");
                const int64_t ncell = L->mesh.ncells;
                if (F->slab.active) {       // distributed fine level: 2:1 nested, addressed through global layers
                    if (lv == 1 && (rc = halo_cells(F, const_cast<double *>(mf_)))) return rc;
                    k_restrict_cells_power_nested3<<<grid_for(ncell), kThreads, 0, st>>>(
                        L->mesh.n[0], L->mesh.n[1], L->mesh.n[2], L->slab.active ? L->slab.crow0 : 0, F->mesh.n[2], F->slab.crow0,
                        L->params[4], mf_, M.m);
                    if (L->slab.active) {
                        if ((rc = halo_cells(L, M.m))) return rc;
                    } else if ((rc = gather_cell_rows(F, M.m, (size_t)L->mesh.n[0] * L->mesh.n[1], L->mesh.n[2]))) return rc;
                } else {
                    k_restrict_cells_power3<<<grid_for(ncell), kThreads, 0, st>>>(lat3_of(F->mesh), lat3_of(L->mesh), L->params[4], mf_, M.m);
                }
                L->launches++;
                L->coef[1] = M.m;
                L->coefn[1] = ncell;
            }
            if (L->family == FEMO_FAMILY_SIMP_Q1) {   // coarse density for the rediscretised stiffness
                const double *mf_ = (lv == 1) ? root->coef[1] : F->mgl.m;
                if (!mf_) return set_err(FEMO_ESTATE, "multigrid setup: density coefficient not set");
                const int64_t ncell = L->mesh.ncells;
                k_restrict_cells_power<<<grid_for(ncell), kThreads, 0, st>>>(Lattice{F->mesh.n[0], F->mesh.n[1]}, Lattice{L->mesh.n[0], L->mesh.n[1]}, L->params[3], mf_, M.m);
                L->launches++;
                L->coef[1] = M.m;
                L->coefn[1] = ncell;
            }
            direct = fp32 && lv < nlev - 1 && lattice_dia_direct(L);
            if (direct) rc = lattice_jacobian(L, nullptr, nullptr, true, L->has_bc);      // no CSR values on DIA-only levels
            else rc = femo_assemble_jacobian(L, L->has_bc ? nullptr : M.vals, L->has_bc ? M.vals : nullptr);
            if (rc) return rc;
        }
        const DevPattern &D = L->dpat[0];
        bool dia_setup = direct;
        if (direct) {
            // nothing to convert
        } else if (fp32 && M.ec && M.k0 && L->coef[1] && lv < nlev - 1) {       // matrix-free V-cycle operator of this level
            const int64_t ncell = L->mesh.ncells;
            k_pow_cells<<<grid_for(ncell), kThreads, 0, st>>>(L->coef[1], L->params[4], M.ec, ncell);
            L->launches++;
        } else if (fp32 && M.vals32 && lv < nlev - 1 && dia_offsets(L, M.dia)) {
            if ((rc = dia_convert(L, lv == 0 ? vperm : nullptr))) return rc;
            dia_setup = true;
        } else if (lv == 0 && vperm) {
            return set_err(FEMO_ESTATE, "multigrid setup: gathered fine-level values need its DIA conversion");
        } else if (fp32 && M.vals32 && lv < nlev - 1) {
            M.dia_valid = false;
            M.dia64_valid = false;
            const int64_t nnz = L->pat[0].nnz;
            k_to_f32<<<(int)std::min<int64_t>((nnz + kThreads - 1) / kThreads, (int64_t)L->num_sms * 16), kThreads, 0, st>>>(M.vals, M.vals32, nnz);
            L->launches++;
        }
        if (lv == nlev - 1) {
            if (n > kMgDenseMax) return set_err(FEMO_ELIMIT, "multigrid: coarsest level too large for the dense solve");
            launch_dense_inverse(D.rowptr, D.col, M.vals, (int)n, M.dense_tmp, M.dense, st);
            L->launches++;
        } else {
            if (!dia_setup) {
                const int g = red_grid(L, n);
                k_diag_gershgorin<<<g, kThreads, 0, st>>>(D.rowptr, D.col, M.vals, M.dinv, n, L->own_off, L->own_off + L->own_n, L->d_partials);
                k_max_finalize<<<1, kThreads, 0, st>>>(L->d_partials, g, L->d_scalars, S_TMP2);
                L->launches += 2;
                FEMO_CHECK_LAUNCH();
            }
            if ((rc = allreduce_scalars(L, S_TMP2, 1, true))) return rc;
            FEMO_CUDA(cudaMemcpyAsync(root->d_scalars + S_MG + npend * kSlots, L->d_scalars + S_TMP2, sizeof(double) * kSlots,
                                      cudaMemcpyDeviceToDevice, st));
            pend[npend++] = L;
            if ((npend == kBatch || g_env.mg_setup_sync_each) && (rc = flush())) return rc;
        }
        FEMO_CHECK_LAUNCH();
    }
    if ((rc = flush())) return rc;
    root->mgprog.dirty = true;       // level bounds changed: the fused coarse V-cycle program is rebuilt on first use
    return FEMO_OK;
}
