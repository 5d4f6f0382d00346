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
    int32_t *rowptr = nullptr, *col = nullptr, *rb = nullptr;
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
    size_t arena_bytes = 0;                 // counted by femo_amg_symbolic
    long long numeric_setups = 0;
};

// The AMG arena's layout walk: maps, values and work vectors of every level, in level order.  Level 0 borrows the
// problem's pattern.  femo_amg_symbolic runs it counting (Arena, common.cuh) to size the arena, femo_amg_attach placing.
static void amg_lay_out(Arena &A, const femo_problem *p, const AmgHier &h, std::vector<AmgLevelDev> &lv) {
    const int nl = (int)h.lv.size();
    lv.assign(nl, AmgLevelDev());
    for (int l = 0; l < nl; ++l) {
        const AmgLevelHost &H = h.lv[l];
        AmgLevelDev &L = lv[l];
        auto F = [&](double *&d, size_t c) { A.take(d, std::max<size_t>(c, 1)); };
        L.n = H.n; L.nnz = H.nnz; L.nc = H.nc; L.nnzP = H.nnzP; L.nnzAP = H.nnzAP;
        if (l == 0) {
            const DevPattern &D = p->dpat[0];
            L.rowptr = D.rowptr; L.col = D.col; L.rb = D.rb; L.nrb = D.nrb;
        } else {
            put(A, L.rowptr, H.rowptr); put(A, L.col, H.col); put(A, L.rb, H.rb); L.nrb = (int)H.rb.size() - 1;
            F(L.vals, H.nnz);
        }
        for (double **v : {&L.dinv, &L.x, &L.b, &L.r, &L.d, &L.q}) F(*v, H.n);
        if (l + 1 < nl) {
            put(A, L.p_rowptr, H.p_rowptr); put(A, L.p_col, H.p_col); put(A, L.p_row, H.p_row); put(A, L.p_rb, H.p_rb);
            L.p_nrb = (int)H.p_rb.size() - 1;
            put(A, L.pp_ptr, H.pp_ptr); put(A, L.pp_src, H.pp_src);
            put(A, L.r_rowptr, H.r_rowptr); put(A, L.r_col, H.r_col); put(A, L.r_perm, H.r_perm); put(A, L.r_rb, H.r_rb);
            L.r_nrb = (int)H.r_rb.size() - 1;
            put(A, L.ap_ptr, H.ap_ptr); put(A, L.ap_ia, H.ap_ia); put(A, L.ap_ib, H.ap_ib);
            put(A, L.ac_ptr, H.ac_ptr); put(A, L.ac_ia, H.ac_ia); put(A, L.ac_ib, H.ac_ib);
            F(L.p_vals, H.nnzP); F(L.r_vals, H.nnzP); F(L.ap_vals, H.nnzAP);
        } else if (H.n <= kMgDenseMax) {
            F(L.dense, (size_t)H.n * H.n); F(L.dense_tmp, (size_t)H.n * H.n);
        }
    }
}

static int amg_attach(femo_problem *p, femo_amg *G, void *d_arena, size_t bytes) {
    G->attached = false;
    Arena A(d_arena, bytes, p->stream);
    amg_lay_out(A, p, G->host, G->lv);
    FEMO_CUDA(cudaStreamSynchronize(p->stream));
    int rc = A.check(G->arena_bytes, "femo_amg_attach");
    if (rc) return rc;
    G->attached = true;
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
