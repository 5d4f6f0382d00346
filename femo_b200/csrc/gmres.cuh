// gmres.cuh -- restarted GMRES(m) for the non-symmetric Jacobians (motor families), right
// preconditioned (Jacobi, Chebyshev polynomial, explicit dense inverse, geometric or algebraic multigrid V-cycle), classical Gram-Schmidt
// with re-orthogonalisation (CGS2: two batched dot passes per iteration, one host read each).
// Together with krylov.cuh this replaces KSP preonly + LU(MUMPS), utils_dolfinx.py:405-408,476-512.
#pragma once
#include "krylov.cuh"

namespace femo {

// partial sums of w . V_i for i < cnt (V column-major, leading dimension ld) over the owned range
__global__ void __launch_bounds__(kThreads)
    k_multidot(const double *__restrict__ V, int64_t ld, int cnt, const double *__restrict__ w, int64_t o0, int64_t o1,
               double *__restrict__ partials) {
    for (int i = 0; i < cnt; ++i) {
        const double *v = V + (int64_t)i * ld;
        double acc = 0.0;
        for (int64_t k = o0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < o1; k += (int64_t)gridDim.x * blockDim.x)
            acc += w[k] * v[k];
        acc = block_sum(acc);
        if (threadIdx.x == 0) partials[(int64_t)i * gridDim.x + blockIdx.x] = acc;
    }
}

__global__ void __launch_bounds__(kThreads) k_finalize_multi(const double *__restrict__ partials, int np, int cnt, double *sc, int slot0) {
    for (int i = 0; i < cnt; ++i) {
        double acc = 0.0;
        for (int k = threadIdx.x; k < np; k += blockDim.x) acc += partials[(int64_t)i * np + k];
        acc = block_sum(acc);
        if (threadIdx.x == 0) sc[slot0 + i] = acc;
    }
}

// w += sign * sum_i sc[slot0+i] V_i
__global__ void __launch_bounds__(kThreads)
    k_lincomb(const double *__restrict__ V, int64_t ld, int cnt, const double *__restrict__ sc, int slot0, double sign,
              double *__restrict__ w, int64_t n) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int i = 0; i < cnt; ++i) acc += sc[slot0 + i] * V[(int64_t)i * ld + k];
        w[k] += sign * acc;
    }
}

__global__ void __launch_bounds__(kThreads) k_scale_to(double a, const double *__restrict__ in, double *__restrict__ out, int64_t n) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) out[k] = a * in[k];
}

}  // namespace femo

using namespace femo;

constexpr int kGmresMax = 72;   // S_GM .. S_GM+kGmresMax scalar slots
static_assert(S_GM + kGmresMax + 1 <= S_MG, "GMRES Hessenberg column overlaps the multigrid set-up slots");

static int gmres_solve(femo_problem *p, const double *vals, const double *b, double *x, femo_krylov_opts o,
                       femo_krylov_info *info) {
    default_krylov(o);
    if (!p->gm_basis) return set_err(FEMO_ESTATE, "GMRES basis not reserved for this problem");
    if (o.precond == 2 && p->mg.empty()) o.precond = 0;
    if (o.precond == 3 && !p->d_dense) o.precond = 0;
    Precond P = precond_params(o, ChebParams{12, 150.0});
    P.mg.ratio = MgParams().ratio;       // under GMRES cheb_ratio sets the polynomial and the AMG smoother, not the V-cycle's
    const int m = (o.restart > 1) ? std::min(o.restart, p->gm_restart) : p->gm_restart;
    const int64_t n = p->state.ndofs, o0 = p->own_off, o1 = p->own_off + p->own_n;
    const DevPattern &D = p->dpat[0];
    cudaStream_t st = p->stream;
    const int g = red_grid(p, n);
    double *V = p->gm_basis, *w = p->kr_q, *z = p->kr_z, *r = p->kr_r, *t = p->kr_p;
    int rc, spmvs = 0, its = 0;
    if ((rc = precond_setup(p, P, vals, p->wk_extra))) return rc;
    double s2;
    if ((rc = norm2_sq(p, b, &s2))) return rc;
    const double bnorm = std::sqrt(s2), tol = std::max(o.rtol * bnorm, o.atol);
    double rnorm = 0.0;
    bool conv = false;
    std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), gvec(m + 1), y(m);
    while (true) {
        if ((rc = launch_spmv<false>(p, D.rb, D.nrb, D.rowptr, D.col, vals, x, r, b, nullptr))) return rc;   // r = b - A x
        ++spmvs;
        if ((rc = norm2_sq(p, r, &s2))) return rc;
        rnorm = std::sqrt(s2);
        if (!(rnorm == rnorm)) break;
        if (rnorm <= tol) { conv = true; break; }
        if (its >= o.max_it) break;
        k_scale_to<<<g, kThreads, 0, st>>>(1.0 / rnorm, r, V, n);
        p->launches++;
        std::fill(H.begin(), H.end(), 0.0);
        std::fill(gvec.begin(), gvec.end(), 0.0);
        gvec[0] = rnorm;
        int j = 0;
        for (; j < m && its < o.max_it; ++j) {
            double *vj = V + (int64_t)j * n, *vn = V + (int64_t)(j + 1) * n;
            if ((rc = precond_apply(p, P, vj, z))) return rc;
            if ((rc = launch_spmv<false>(p, D.rb, D.nrb, D.rowptr, D.col, vals, z, w, nullptr, nullptr))) return rc;
            ++spmvs;
            for (int pass = 0; pass < 2; ++pass) {          // CGS2
                k_multidot<<<g, kThreads, 0, st>>>(V, n, j + 1, w, o0, o1, p->d_partials_big);
                k_finalize_multi<<<1, kThreads, 0, st>>>(p->d_partials_big, g, j + 1, p->d_scalars, S_GM);
                p->launches += 2;
                if ((rc = allreduce_scalars(p, S_GM, j + 1))) return rc;
                k_lincomb<<<g, kThreads, 0, st>>>(V, n, j + 1, p->d_scalars, S_GM, -1.0, w, n);
                p->launches++;
                FEMO_CHECK_LAUNCH();
                double hcol[kGmresMax + 1];
                if ((rc = read_scalars(p, S_GM, j + 1, hcol))) return rc;
                for (int i = 0; i <= j; ++i) H[(size_t)i * m + j] += hcol[i];
            }
            if ((rc = norm2_sq(p, w, &s2))) return rc;
            const double hn = std::sqrt(s2);
            H[(size_t)(j + 1) * m + j] = hn;
            if (hn > 0.0) {
                k_scale_to<<<g, kThreads, 0, st>>>(1.0 / hn, w, vn, n);
                p->launches++;
            }
            // Givens rotations on column j
            for (int i = 0; i < j; ++i) {
                const double a = H[(size_t)i * m + j], c = H[(size_t)(i + 1) * m + j];
                H[(size_t)i * m + j] = cs[i] * a + sn[i] * c;
                H[(size_t)(i + 1) * m + j] = -sn[i] * a + cs[i] * c;
            }
            const double a = H[(size_t)j * m + j], c = H[(size_t)(j + 1) * m + j], den = std::hypot(a, c);
            cs[j] = den > 0 ? a / den : 1.0;
            sn[j] = den > 0 ? c / den : 0.0;
            H[(size_t)j * m + j] = den;
            H[(size_t)(j + 1) * m + j] = 0.0;
            gvec[j + 1] = -sn[j] * gvec[j];
            gvec[j] = cs[j] * gvec[j];
            ++its;
            rnorm = std::fabs(gvec[j + 1]);
            if (rnorm <= tol || hn == 0.0) { ++j; break; }
        }
        // y = H^-1 g ; x += M^-1 (V y)
        for (int i = j - 1; i >= 0; --i) {
            double sacc = gvec[i];
            for (int k = i + 1; k < j; ++k) sacc -= H[(size_t)i * m + k] * y[k];
            y[i] = sacc / H[(size_t)i * m + i];
        }
        for (int i = 0; i < j; ++i) p->h_pinned[i] = y[i];
        FEMO_CUDA(cudaMemcpyAsync(p->d_scalars + S_GM, p->h_pinned, sizeof(double) * j, cudaMemcpyHostToDevice, st));
        FEMO_CUDA(cudaMemsetAsync(t, 0, sizeof(double) * n, st));
        k_lincomb<<<g, kThreads, 0, st>>>(V, n, j, p->d_scalars, S_GM, 1.0, t, n);
        p->launches++;
        if ((rc = precond_apply(p, P, t, z))) return rc;
        k_axpy<<<g, kThreads, 0, st>>>(1.0, z, x, n);
        p->launches++;
        FEMO_CHECK_LAUNCH();
        FEMO_CUDA(cudaStreamSynchronize(st));   // h_pinned is reused by the next read
    }
    if ((rc = halo_nodes(p, x))) return rc;
    if (info) {
        info->iterations = its;
        info->converged = conv ? 1 : 0;
        info->rnorm = rnorm;
        info->bnorm = bnorm;
        info->spmv_count = spmvs;
    }
    return FEMO_OK;
}
