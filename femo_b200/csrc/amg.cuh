// amg.cuh -- device side of the smoothed-aggregation preconditioner (precond 4) for problems without a lattice
// hierarchy: unstructured meshes, the motor annulus with its tagged subdomains.  Pattern phase: amg_setup.cpp (host,
// once per pattern).  Numeric phase (here, once per Jacobian): per level one Gershgorin / diagonal pass and three sorted
// segmented reductions (prolongator, A P, P^T A P) over the index lists of the pattern phase -- no atomics, fixed
// summation order.  Solve phase: V-cycle whose every operator application is the CSR-stream SpMV of engine.cu with the
// Chebyshev-Jacobi epilogues the geometric hierarchy uses; restriction and prolongation are SpMVs with R = P^T and P.
// Replaces, together with krylov.cuh / gmres.cuh, KSP preonly + LU(MUMPS) (utils_dolfinx.py:405-408,476-512).
#pragma once
#include "amg_setup.hpp"
#include "common.cuh"

namespace femo {

// P[t] = sum over the A entries k of row(t) whose column lies in aggregate col(t) of (delta - omega a_k / a_rr)
__global__ void __launch_bounds__(kThreads)
    k_amg_prolongator(const int32_t *__restrict__ pp_ptr, const int32_t *__restrict__ pp_src, const int32_t *__restrict__ p_row,
                      const int32_t *__restrict__ col, const double *__restrict__ vals, const double *__restrict__ dinv,
                      const double *__restrict__ scalars, int lmax_slot, double omega_scale, double *__restrict__ p_vals,
                      int64_t nnzP) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= nnzP) return;
    const int32_t r = p_row[t];
    const double w = omega_scale * (4.0 / (3.0 * scalars[lmax_slot])) * dinv[r];
    double acc = 0.0;
    for (int32_t s = pp_ptr[t]; s < pp_ptr[t + 1]; ++s) {
        const int32_t k = pp_src[s];
        acc += (col[k] == r ? 1.0 : 0.0) - w * vals[k];
    }
    p_vals[t] = acc;
}

// out[t] = sum_{s in [ptr[t], ptr[t+1])} X[ia[s]] * Y[ib[s]]   (sources ascending: deterministic)
__global__ void __launch_bounds__(kThreads)
    k_pair_segreduce(const int32_t *__restrict__ ptr, const int32_t *__restrict__ ia, const int32_t *__restrict__ ib,
                     const double *__restrict__ X, const double *__restrict__ Y, double *__restrict__ out, int64_t n) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    double acc = 0.0;
    for (int32_t s = ptr[t]; s < ptr[t + 1]; ++s) acc += X[ia[s]] * Y[ib[s]];
    out[t] = acc;
}

}  // namespace femo

using namespace femo;

struct AmgLevelDev {
    int64_t n = 0, nnz = 0, nc = 0, nnzP = 0, nnzAP = 0;
    const int32_t *rowptr = nullptr, *col = nullptr, *rb = nullptr;
    int nrb = 0;
    double *vals = nullptr;                 // level 0: the matrix of the current solve (not owned)
    double *dinv = nullptr, *x = nullptr, *b = nullptr, *r = nullptr, *d = nullptr, *q = nullptr;
    double lmax = 2.0;
    int32_t *p_rowptr = nullptr, *p_col = nullptr, *p_row = nullptr, *p_rb = nullptr, *pp_ptr = nullptr, *pp_src = nullptr;
    int32_t *r_rowptr = nullptr, *r_col = nullptr, *r_perm = nullptr, *r_rb = nullptr;
    int32_t *ap_ptr = nullptr, *ap_ia = nullptr, *ap_ib = nullptr, *ac_ptr = nullptr, *ac_ia = nullptr, *ac_ib = nullptr;
    int p_nrb = 0, r_nrb = 0;
    double *p_vals = nullptr, *r_vals = nullptr, *ap_vals = nullptr;
    double *dense = nullptr, *dense_tmp = nullptr;
    bool halo = false;                      // level 0 of an unstructured partition: refresh the ghost dofs before every operator application
};

struct femo_amg {
    AmgHier host;
    std::vector<AmgLevelDev> lv;
    bool attached = false;
    size_t arena_bytes = 0;
    long long numeric_setups = 0;
};

// bytes of device memory the hierarchy needs (maps + values + work vectors of every level)
static size_t amg_arena_bytes(const AmgHier &h) {
    size_t w = 0;
    const int nl = (int)h.lv.size();
    for (int l = 0; l < nl; ++l) {
        const AmgLevelHost &L = h.lv[l];
        auto I = [&](size_t c) { w += Arena::need(std::max<size_t>(c, 1), 4); };
        auto F = [&](size_t c) { w += Arena::need(std::max<size_t>(c, 1), 8); };
        if (l > 0) { I(L.n + 1); I(L.nnz); I(L.rb.size()); F(L.nnz); }
        F(L.n); F(L.n); F(L.n); F(L.n); F(L.n); F(L.n);                     // dinv, x, b, r, d, q
        if (l + 1 < nl) {
            I(L.n + 1); I(L.nnzP); I(L.nnzP); I(L.p_rb.size()); I(L.nnzP + 1); I(L.pp_src.size());
            I(L.nc + 1); I(L.nnzP); I(L.nnzP); I(L.r_rb.size());
            I(L.nnzAP + 1); I(L.ap_ia.size()); I(L.ap_ib.size());
            I(L.nnzC + 1); I(L.ac_ia.size()); I(L.ac_ib.size());
            F(L.nnzP); F(L.nnzP); F(L.nnzAP);
        } else if (L.n <= kMgDenseMax) {
            F((size_t)L.n * L.n); F((size_t)L.n * L.n);
        }
    }
    return w + 4096;
}

static int amg_attach(femo_problem *p, femo_amg *G, void *d_arena, size_t bytes) {
    Arena A;
    A.reset(d_arena, bytes);
    cudaStream_t st = p->stream;
    const int nl = (int)G->host.lv.size();
    G->lv.assign(nl, AmgLevelDev());
    bool ok = true;
    auto upI = [&](const std::vector<int32_t> &v) -> int32_t * {
        int32_t *d = A.take<int32_t>(std::max<size_t>(v.size(), 1));
        if (!d) { ok = false; return nullptr; }
        if (!v.empty()) cudaMemcpyAsync(d, v.data(), v.size() * 4, cudaMemcpyHostToDevice, st);
        return d;
    };
    auto F = [&](size_t c) -> double * {
        double *d = A.take<double>(std::max<size_t>(c, 1));
        if (!d) ok = false;
        return d;
    };
    for (int l = 0; l < nl && ok; ++l) {
        const AmgLevelHost &H = G->host.lv[l];
        AmgLevelDev &L = G->lv[l];
        L.n = H.n; L.nnz = H.nnz; L.nc = H.nc; L.nnzP = H.nnzP; L.nnzAP = H.nnzAP;
        if (l == 0) {
            const DevPattern &D = p->dpat[0];
            L.rowptr = D.rowptr; L.col = D.col; L.rb = D.rb; L.nrb = D.nrb;
        } else {
            L.rowptr = upI(H.rowptr); L.col = upI(H.col); L.rb = upI(H.rb); L.nrb = (int)H.rb.size() - 1;
            L.vals = F(H.nnz);
        }
        L.dinv = F(H.n); L.x = F(H.n); L.b = F(H.n); L.r = F(H.n); L.d = F(H.n); L.q = F(H.n);
        if (l + 1 < nl) {
            L.p_rowptr = upI(H.p_rowptr); L.p_col = upI(H.p_col); L.p_row = upI(H.p_row); L.p_rb = upI(H.p_rb);
            L.p_nrb = (int)H.p_rb.size() - 1;
            L.pp_ptr = upI(H.pp_ptr); L.pp_src = upI(H.pp_src);
            L.r_rowptr = upI(H.r_rowptr); L.r_col = upI(H.r_col); L.r_perm = upI(H.r_perm); L.r_rb = upI(H.r_rb);
            L.r_nrb = (int)H.r_rb.size() - 1;
            L.ap_ptr = upI(H.ap_ptr); L.ap_ia = upI(H.ap_ia); L.ap_ib = upI(H.ap_ib);
            L.ac_ptr = upI(H.ac_ptr); L.ac_ia = upI(H.ac_ia); L.ac_ib = upI(H.ac_ib);
            L.p_vals = F(H.nnzP); L.r_vals = F(H.nnzP); L.ap_vals = F(H.nnzAP);
        } else if (H.n <= kMgDenseMax) {
            L.dense = F((size_t)H.n * H.n); L.dense_tmp = F((size_t)H.n * H.n);
        }
    }
    FEMO_CUDA(cudaStreamSynchronize(st));
    if (!ok) return set_err(FEMO_EINVAL, "femo_amg_attach: arena smaller than femo_amg_symbolic reported");
    G->attached = true;
    G->arena_bytes = bytes;
    return FEMO_OK;
}

// one operator application of a level with the epilogue `epi` (CSR-stream SpMV of engine.cu)
static int amg_apply(femo_problem *p, const int32_t *rb, int nrb, const int32_t *rowptr, const int32_t *col, const double *vals,
                     int epi, const double *x, double *y, const SpmvEpi &E, bool halo = false) {
    if (halo) {
        int rc = halo_nodes(p, const_cast<double *>(x));
        if (rc) return rc;
    }
    const int grid = spmv_grid(p, nrb);
    cudaStream_t st = p->stream;
    if (epi == EPI_PLAIN) k_spmv<false, EPI_PLAIN, double><<<grid, kThreads, 0, st>>>(rb, nrb, rowptr, col, vals, x, y, E, nullptr);
    else if (epi == EPI_CHEB0) k_spmv<false, EPI_CHEB0, double><<<grid, kThreads, 0, st>>>(rb, nrb, rowptr, col, vals, x, y, E, nullptr);
    else if (epi == EPI_CHEBK) k_spmv<false, EPI_CHEBK, double><<<grid, kThreads, 0, st>>>(rb, nrb, rowptr, col, vals, x, y, E, nullptr);
    else k_spmv<false, EPI_ADD, double><<<grid, kThreads, 0, st>>>(rb, nrb, rowptr, col, vals, x, y, E, nullptr);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// numeric phase: every level's diagonal / Gershgorin bound, prolongator, restriction and Galerkin operator from `vals`
static int amg_numeric(femo_problem *p, femo_amg *G, const double *vals) {
    if (!G || !G->attached) return set_err(FEMO_ESTATE, "precond 4 (AMG) needs femo_amg_symbolic + femo_amg_attach first");
    if (p->slab.active) return set_err(FEMO_ESTATE, "slab problems use the lattice hierarchy, not the AMG preconditioner");
    cudaStream_t st = p->stream;
    const int nl = (int)G->lv.size();
    G->lv[0].vals = const_cast<double *>(vals);
    // Unstructured partition: level 0 is the distributed operator itself (its smoother exchanges halos and uses the global
    // Gershgorin bound, so every rank runs the same Chebyshev polynomial on its owned rows); the coarse correction is local
    // to the rank -- ghost rows have empty prolongator rows, so they neither restrict nor receive corrections: a symmetric
    // two-level additive-in-the-coarse-space preconditioner without communication below level 0.
    G->lv[0].halo = p->gpart.active;
    int rc;
    for (int l = 0; l < nl; ++l) {
        AmgLevelDev &L = G->lv[l];
        const int g = red_grid(p, L.n);
        k_diag_gershgorin<<<g, kThreads, 0, st>>>(L.rowptr, L.col, L.vals, L.dinv, L.n, 0, L.n, p->d_partials);
        k_max_finalize<<<1, kThreads, 0, st>>>(p->d_partials, g, p->d_scalars, S_GM + l);
        p->launches += 2;
        if (l == 0 && p->gpart.active && (rc = allreduce_scalars(p, S_GM, 1, true))) return rc;
        if (l + 1 < nl) {
            AmgLevelDev &C = G->lv[l + 1];
            k_amg_prolongator<<<grid_for(L.nnzP), kThreads, 0, st>>>(L.pp_ptr, L.pp_src, L.p_row, L.col, L.vals, L.dinv, p->d_scalars,
                                                                      S_GM + l, G->host.opts.omega_scale, L.p_vals, L.nnzP);
            k_permute<<<grid_for(L.nnzP), kThreads, 0, st>>>(L.r_perm, L.p_vals, L.r_vals, L.nnzP);
            k_pair_segreduce<<<grid_for(L.nnzAP), kThreads, 0, st>>>(L.ap_ptr, L.ap_ia, L.ap_ib, L.vals, L.p_vals, L.ap_vals, L.nnzAP);
            k_pair_segreduce<<<grid_for(C.nnz), kThreads, 0, st>>>(L.ac_ptr, L.ac_ia, L.ac_ib, L.p_vals, L.ap_vals, C.vals, C.nnz);
            p->launches += 4;
        } else if (L.dense) {
            k_dense_inverse<<<1, kThreads, 0, st>>>(L.rowptr, L.col, L.vals, (int)L.n, L.dense_tmp, L.dense);
            p->launches++;
        }
        FEMO_CHECK_LAUNCH();
    }
    double lm[32];
    if ((rc = read_scalars(p, S_GM, nl, lm))) return rc;      // one synchronisation for the Chebyshev bounds of all levels
    for (int l = 0; l < nl; ++l) G->lv[l].lmax = lm[l];
    G->numeric_setups++;
    return FEMO_OK;
}

// Chebyshev-Jacobi smoother of degree deg on [lmax/ratio, lmax], every operator application a CSR-stream SpMV
static int amg_smooth(femo_problem *p, AmgLevelDev &L, const double *b, double *x, bool zero_guess, int deg, double ratio) {
    return cheb_smooth(p, ChebWork{L.dinv, L.r, L.d, L.q, L.n, L.lmax}, b, x, zero_guess, deg, ratio, false,
                       [&](int kind, const double *xin, const SpmvEpi &E) {
                           return amg_apply(p, L.rb, L.nrb, L.rowptr, L.col, L.vals, kind, xin, nullptr, E, L.halo);
                       });
}

// one V-cycle from a zero initial guess: x ~ A_l^-1 b
static int amg_vcycle(femo_problem *p, femo_amg *G, int l, const double *b, double *x, const ChebParams &ap) {
    AmgLevelDev &L = G->lv[l];
    cudaStream_t st = p->stream;
    int rc;
    if (l + 1 == (int)G->lv.size()) {
        if (L.dense) {
            k_dense_apply<<<(int)((L.n * 32 + kThreads - 1) / kThreads), kThreads, 0, st>>>(L.dense, b, x, (int)L.n);
            p->launches++;
            FEMO_CHECK_LAUNCH();
            return FEMO_OK;
        }
        return amg_smooth(p, L, b, x, true, 12, 30.0);       // coarsening stalled above the dense limit
    }
    AmgLevelDev &C = G->lv[l + 1];
    if ((rc = amg_smooth(p, L, b, x, true, ap.degree, ap.ratio))) return rc;
    SpmvEpi E;
    E.b = b;
    if ((rc = amg_apply(p, L.rb, L.nrb, L.rowptr, L.col, L.vals, EPI_PLAIN, x, L.r, E, L.halo))) return rc;            // r = b - A x
    if ((rc = amg_apply(p, L.r_rb, L.r_nrb, L.r_rowptr, L.r_col, L.r_vals, EPI_PLAIN, L.r, C.b, SpmvEpi()))) return rc;   // bc = P^T r
    if ((rc = amg_vcycle(p, G, l + 1, C.b, C.x, ap))) return rc;
    if ((rc = amg_apply(p, L.p_rb, L.p_nrb, L.p_rowptr, L.p_col, L.p_vals, EPI_ADD, C.x, x, SpmvEpi()))) return rc;       // x += P xc
    return amg_smooth(p, L, b, x, false, ap.degree, ap.ratio);
}
