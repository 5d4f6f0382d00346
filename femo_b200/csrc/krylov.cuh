// krylov.cuh -- CG drivers (K8/K9): Jacobi-preconditioned CG with fused vector
// kernels, and PCG with a multigrid V-cycle or an explicit dense inverse as
// preconditioner.  They replace KSP preonly + LU(MUMPS) of the reference
// (femo/fea/utils_dolfinx.py:405-408,476-512).
//
// Scalars (alpha, beta, r.z, ...) live on the device; partial sums are reduced in
// a fixed order; on several GPUs the reductions run over each rank's OWNED dofs
// and are combined with ncclAllReduce on the same stream -- the host only reads
// the residual norm every `check_every` iterations.
#pragma once
#include "common.cuh"
#include "dist_ops.cuh"

namespace femo {

__device__ __forceinline__ bool owned(int64_t i, int64_t o0, int64_t o1) { return i >= o0 && i < o1; }

// r = b - q ; p = dinv*r ; partials of r.(dinv r), r.r over the owned range
__global__ void __launch_bounds__(kThreads)
    k_cg_init(const double *__restrict__ b, const double *__restrict__ q, const double *__restrict__ dinv,
              double *__restrict__ r, double *__restrict__ p, int64_t n, int64_t o0, int64_t o1,
              double *__restrict__ prz, double *__restrict__ prr) {
    double rz = 0.0, rr = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double ri = b[i] - q[i];
        const double zi = dinv[i] * ri;
        r[i] = ri;
        p[i] = zi;
        if (owned(i, o0, o1)) {
            rz += ri * zi;
            rr += ri * ri;
        }
    }
    rz = block_sum(rz);
    rr = block_sum(rr);
    if (threadIdx.x == 0) {
        prz[blockIdx.x] = rz;
        prr[blockIdx.x] = rr;
    }
}

// x += alpha p ; r -= alpha q ; partials of r.(dinv r) [dinv may be null] and r.r
__global__ void __launch_bounds__(kThreads)
    k_cg_update(const double *__restrict__ sc, const double *__restrict__ p, const double *__restrict__ q,
                const double *__restrict__ dinv, double *__restrict__ x, double *__restrict__ r, int64_t n, int64_t o0,
                int64_t o1, double *__restrict__ prz, double *__restrict__ prr) {
    const double alpha = sc[S_ALPHA];
    double rz = 0.0, rr = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        x[i] += alpha * p[i];
        const double ri = r[i] - alpha * q[i];
        r[i] = ri;
        if (owned(i, o0, o1)) {
            if (dinv) rz += ri * ri * dinv[i];
            rr += ri * ri;
        }
    }
    rr = block_sum(rr);
    if (dinv) rz = block_sum(rz);
    if (threadIdx.x == 0) {
        if (dinv) prz[blockIdx.x] = rz;
        prr[blockIdx.x] = rr;
    }
}

// p = z + beta p with z = dinv*r (Jacobi, zvec null) or z = zvec; first: p = z
__global__ void __launch_bounds__(kThreads)
    k_cg_dir(const double *__restrict__ sc, const double *__restrict__ r, const double *__restrict__ dinv,
             const double *__restrict__ zvec, double *__restrict__ p, int64_t n, int first) {
    const double beta = first ? 0.0 : sc[S_BETA];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double zi = zvec ? zvec[i] : dinv[i] * r[i];
        p[i] = zi + beta * p[i];
    }
}

// r = b - q ; partial r.r over the owned range
__global__ void __launch_bounds__(kThreads)
    k_residual_rr(const double *__restrict__ b, const double *__restrict__ q, double *__restrict__ r, int64_t n,
                  int64_t o0, int64_t o1, double *__restrict__ prr) {
    double rr = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double ri = b[i] - q[i];
        r[i] = ri;
        if (owned(i, o0, o1)) rr += ri * ri;
    }
    rr = block_sum(rr);
    if (threadIdx.x == 0) prr[blockIdx.x] = rr;
}

// one CTA: fixed-order sums of two partial arrays -> scalars[slotA], scalars[slotB] (pb may be null)
__global__ void __launch_bounds__(kThreads)
    k_finalize2(const double *__restrict__ pa, const double *__restrict__ pb, int np, double *sc, int slotA, int slotB) {
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < np; i += blockDim.x) {
        a += pa[i];
        if (pb) b += pb[i];
    }
    a = block_sum(a);
    b = block_sum(b);
    if (threadIdx.x == 0) {
        sc[slotA] = a;
        if (pb) sc[slotB] = b;
    }
}

// scalar recurrences on already (all-)reduced values
//   op 0: alpha = rz / pq
//   op 1: beta = tmp0 / rz ; rz = tmp0 ; rr = tmp1
//   op 2: beta = tmp0 / rz ; rz = tmp0
//   op 3: rz = tmp0
__global__ void k_scalar_op(double *sc, int op) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (op == 0) {
        sc[S_ALPHA] = (sc[S_PQ] != 0.0) ? sc[S_RZ] / sc[S_PQ] : 0.0;
    } else if (op == 1 || op == 2) {
        sc[S_BETA] = (sc[S_RZ] != 0.0) ? sc[S_TMP0] / sc[S_RZ] : 0.0;
        sc[S_RZ] = sc[S_TMP0];
        if (op == 1) sc[S_RR] = sc[S_TMP1];
    } else {
        sc[S_RZ] = sc[S_TMP0];
    }
}

__global__ void __launch_bounds__(kThreads) k_hadamard(const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ out, int64_t n) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) out[k] = a[k] * b[k];
}

}  // namespace femo

using namespace femo;

// fine-level rows up to which the PCG iteration is replayed as a CUDA graph (FEMO_GRAPH_MAX_ROWS overrides)
static int64_t graph_max_rows() { return g_env.graph_max_rows; }

// Runs a solve on the problem's side stream: fork behind the caller's stream on construction, join on destruction.
struct StreamSwap {
    femo_problem *p;
    cudaStream_t old = nullptr;
    bool active = false;
    StreamSwap(femo_problem *p_, bool on) : p(p_) {
        if (!on || p->stream == p->stream2) return;
        old = p->stream;
        if (cudaEventRecord(p->ev_fork, old) != cudaSuccess || cudaStreamWaitEvent(p->stream2, p->ev_fork, 0) != cudaSuccess) {
            cudaGetLastError();
            return;
        }
        set(p->stream2);
        active = true;
    }
    void set(cudaStream_t s) {
        p->stream = s;
        for (femo_problem *c : p->mg) c->stream = s;
    }
    ~StreamSwap() {
        if (!active) return;
        cudaEventRecord(p->ev_join, p->stream2);
        cudaStreamWaitEvent(old, p->ev_join, 0);
        set(old);
    }
};

static void default_krylov(femo_krylov_opts &o) {
    if (o.rtol <= 0) o.rtol = 1e-10;
    if (o.atol < 0) o.atol = 0;
    if (o.max_it <= 0) o.max_it = 100000;
    if (o.check_every <= 0) o.check_every = 1;
}

// sum of partials -> scalar slot(s) -> all ranks
static int reduce_to(femo_problem *p, const double *pa, const double *pb, int np, int slotA, int slotB) {
    if (g_link.active && g_comm.active && partitioned(p) && (!pb || slotB == slotA + 1)) {
        // block sums of the partials and the all-reduce over the ranks in ONE kernel (link.cuh)
        const unsigned int seq = ++g_link.seq_ar;
        k_link_allreduce<<<1, kThreads, 0, p->stream>>>(g_link.dev(), p->d_scalars, pb ? 2 : 1, 0, pa, pb, np, slotA, slotB, seq);
        p->launches++;
        g_comm.allreduces++;
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    }
    k_finalize2<<<1, kThreads, 0, p->stream>>>(pa, pb, np, p->d_scalars, slotA, slotB);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    if (pb && slotB == slotA + 1) return allreduce_scalars(p, slotA, 2);
    int rc = allreduce_scalars(p, slotA, 1);
    if (rc || !pb) return rc;
    return allreduce_scalars(p, slotB, 1);
}

static int scalar_op(femo_problem *p, int op) {
    k_scalar_op<<<1, 32, 0, p->stream>>>(p->d_scalars, op);
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// ||a||^2 over the owned dofs of all ranks -> host
static int norm2_sq(femo_problem *p, const double *a, double *out) {
    const int64_t n = p->own_n;
    int g = red_grid(p, n);
    k_dot<<<g, kThreads, 0, p->stream>>>(a + p->own_off, a + p->own_off, n, p->d_partials);
    p->launches++;
    int rc;
    if ((rc = reduce_to(p, p->d_partials, nullptr, g, S_TMP0, 0))) return rc;
    return read_scalars(p, S_TMP0, 1, out);
}

// Gershgorin bound + inverse diagonal of level 0 for the Chebyshev polynomial preconditioner (precond 1)
static int cheb_setup(femo_problem *p, const double *vals) {
    const int64_t n = p->state.ndofs;
    const DevPattern &D = p->dpat[0];
    const int g = red_grid(p, n);
    int rc;
    p->mgl.vals = const_cast<double *>(vals);
    k_diag_gershgorin<<<g, kThreads, 0, p->stream>>>(D.rowptr, D.col, vals, p->mgl.dinv, n, p->own_off, p->own_off + p->own_n, p->d_partials);
    k_max_finalize<<<1, kThreads, 0, p->stream>>>(p->d_partials, g, p->d_scalars, S_TMP2);
    p->launches += 2;
    FEMO_CHECK_LAUNCH();
    if ((rc = allreduce_scalars(p, S_TMP2, 1, true))) return rc;
    return read_scalars(p, S_TMP2, 1, &p->mgl.lmax);
}

// Preconditioner of the Krylov drivers (CG and GMRES):
//   precond 0: Jacobi, 1: Chebyshev polynomial, 2: geometric multigrid V-cycle, 3: explicit dense inverse,
//   4: smoothed-aggregation AMG V-cycle (amg.cuh)
struct Precond {
    int pre = 0;
    MgParams mg;           // precond 2
    ChebParams amg;        // precond 4
    ChebParams poly;       // precond 1: the polynomial on the root, fp64 CSR
};

// cheb_degree / cheb_ratio of the options override the smoother defaults; `poly`: the solver's own default polynomial
static Precond precond_params(const femo_krylov_opts &o, ChebParams poly) {
    Precond P;
    P.pre = o.precond;
    P.mg.fp32 = (o.mg_precision == 0);
    if (o.cheb_degree > 0) P.mg.degree = P.amg.degree = poly.degree = o.cheb_degree;
    if (o.cheb_ratio > 1.0) P.mg.ratio = P.amg.ratio = poly.ratio = o.cheb_ratio;
    P.poly = poly;
    return P;
}

// set-up for the matrix `vals`.  q: the root's fourth V-cycle work vector (GMRES keeps kr_q for itself);
// dia_prepared: `vals` was assembled with the fine level's DIA planes (mg_setup's level0_dia)
// vperm: the matrix is vals[vperm[t]] (multigrid only, see level0_dia_only)
static int precond_setup(femo_problem *p, const Precond &P, const double *vals, double *q, bool dia_prepared = false,
                         const int32_t *vperm = nullptr) {
    const int64_t n = p->state.ndofs;
    const DevPattern &D = p->dpat[0];
    cudaStream_t st = p->stream;
    int rc;
    p->mgl.dinv = p->kr_dinv;
    p->mgl.r = p->kr_w;
    p->mgl.d = p->kr_d;
    p->mgl.q = q;
    if (P.pre == 2) {
        if ((rc = mg_setup(p, vals, P.mg.fp32, dia_prepared, vperm))) return rc;
    } else if (vperm) {
        return set_err(FEMO_ESTATE, "gathered values need the multigrid preconditioner");
    } else if (P.pre == 4) {
        if ((rc = amg_numeric(p, p->amg, vals))) return rc;
    } else if (P.pre == 1) {
        if ((rc = cheb_setup(p, vals))) return rc;
    } else if (P.pre == 3) {
        launch_dense_inverse(D.rowptr, D.col, vals, (int)n, p->d_dense_tmp, p->d_dense, st);
        p->launches++;
    } else {
        k_diag_inv<<<grid_for(n), kThreads, 0, st>>>(D.rowptr, D.col, vals, p->kr_dinv, n);
        p->launches++;
    }
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// out = M^-1 in.  Jacobi is GMRES's: CG folds it into k_cg_init / k_cg_update.
static int precond_apply(femo_problem *p, const Precond &P, const double *in, double *out) {
    const int64_t n = p->state.ndofs;
    cudaStream_t st = p->stream;
    switch (P.pre) {
        case 1: return mg_smooth(p, in, out, true, P.poly.degree, P.poly.ratio, false);
        case 2: return mg_vcycle(p, 0, in, out, P.mg);
        case 4: return amg_vcycle(p, p->amg, 0, in, out, P.amg);
        case 3: k_dense_apply<<<(int)((n * 32 + kThreads - 1) / kThreads), kThreads, 0, st>>>(p->d_dense, in, out, (int)n); break;
        default: k_hadamard<<<red_grid(p, n), kThreads, 0, st>>>(p->kr_dinv, in, out, n); break;
    }
    p->launches++;
    FEMO_CHECK_LAUNCH();
    return FEMO_OK;
}

// Preconditioned CG on the dR/du pattern; `vals` already in the layout to multiply with.  Preconditioner: Precond.
// op_current: the caller guarantees that `vals` is the (BC'd) Jacobian of the coefficients currently bound to the
// problem (true inside femo_newton_solve, which assembles it itself): hexahedral lattices then apply the operator
// matrix-free in the recurrence too.  Matrices handed in through femo_linear_solve are always streamed as given.
static int cg_solve(femo_problem *p, const double *vals, const double *b, double *x, femo_krylov_opts o,
                    femo_krylov_info *info, bool op_current = false, bool dia_prepared = false,
                    const int32_t *vperm = nullptr) {
    default_krylov(o);
    if (o.precond == 2 && p->mg.empty()) o.precond = 0;
    if (o.precond == 3 && !p->d_dense) return set_err(FEMO_ELIMIT, "precond 3 (dense direct) needs N <= 512 on one GPU");
    const Precond P = precond_params(o, ChebParams{8, 60.0});
    const int pre = P.pre;
    const int64_t n = p->state.ndofs, o0 = p->own_off, o1 = p->own_off + p->own_n;
    const DevPattern &D = p->dpat[0];
    // Launch-bound problems replay the PCG iteration from a CUDA graph (below).  The legacy default stream cannot be
    // captured, so such a solve runs on the problem's own side stream, ordered after / before the caller's stream by events.
    const bool use_graph = !g_comm.active && pre == 2 && !g_env.no_graph && (n <= graph_max_rows() || g_env.force_graph);
    StreamSwap swap(p, use_graph && p->stream2);
    cudaStream_t st = p->stream;
    double *pa = p->d_partials, *pb = p->d_partials + kMaxPartials;
    const int g = red_grid(p, n), go = red_grid(p, p->own_n);
    int rc, np = 0, spmvs = 0;
    if ((rc = precond_setup(p, P, vals, p->kr_q, dia_prepared, vperm))) return rc;
    // ||b||^2
    k_dot<<<go, kThreads, 0, st>>>(b + p->own_off, b + p->own_off, p->own_n, pa);
    p->launches++;
    if ((rc = reduce_to(p, pa, nullptr, go, S_BB, 0))) return rc;
    // multigrid: replace the caller's initial guess by the full-multigrid iterate (discretisation accuracy)
    // full-multigrid start (halves the iteration count here; measured on slabs too: 14 vs 27 iterations per step at N=2)
    if (pre == 2 && o.restart != 1 && (rc = mg_fmg(p, b, x, P.mg))) return rc;
    const LevelOp vop = level_op(p, P.mg.fp32);
    const bool mf_outer = op_current && pre == 2 && vop == LevelOp::MATFREE;
    const bool dia_outer = pre == 2 && p->mgl.dia64_valid && vop == LevelOp::DIA;       // fp64 planes of `vals` (set-up)
    const bool bsr_outer = !mf_outer && !dia_outer && bsr3_ready(p);                     // vector states in 3-D: 3x3 blocks
    if (vperm && !dia_outer) return set_err(FEMO_ESTATE, "gathered values need the fp64 DIA planes for the recurrence");
    if (bsr_outer && (rc = bsr3_convert(p, vals))) return rc;
    // q = A xin with the recurrence's operator; dot = std::true_type: also the partial sums of xin.q, their count into np
    auto outer = [&](auto dot, const double *xin, double *q) -> int {
        constexpr bool DOT = decltype(dot)::value;
        int *npo = DOT ? &np : nullptr;
        if (mf_outer) {
            SpmvEpi E0;
            const int r = launch_hex_matfree(p, EPI_PLAIN, xin, q, E0);
            if (r || !DOT) return r;
            k_dot<<<go, kThreads, 0, st>>>(xin + p->own_off, q + p->own_off, p->own_n, p->d_partials);
            p->launches++;
            np = go;
            return FEMO_OK;
        }
        if (dia_outer) return launch_dia64<DOT>(p, xin, q, nullptr, npo);
        if (bsr_outer) return launch_spmv_bsr3<DOT>(p, xin, q, nullptr, npo);
        return launch_spmv<DOT>(p, D.rb, D.nrb, D.rowptr, D.col, vals, xin, q, nullptr, npo);
    };
    // r = b - A x
    if ((rc = outer(std::false_type{}, x, p->kr_q))) return rc;
    ++spmvs;
    if (pre == 0) {
        k_cg_init<<<g, kThreads, 0, st>>>(b, p->kr_q, p->kr_dinv, p->kr_r, p->kr_p, n, o0, o1, pa, pb);
        p->launches++;
        if ((rc = reduce_to(p, pa, pb, g, S_RZ, S_RR))) return rc;
    } else {
        k_residual_rr<<<g, kThreads, 0, st>>>(b, p->kr_q, p->kr_r, n, o0, o1, pb);
        p->launches++;
        if ((rc = reduce_to(p, pb, nullptr, g, S_RR, 0))) return rc;
    }
    FEMO_CHECK_LAUNCH();
    double h[2];
    if ((rc = read_scalars(p, S_RR, 1, &h[0]))) return rc;
    if ((rc = read_scalars(p, S_BB, 1, &h[1]))) return rc;
    const double bnorm = std::sqrt(h[1]);
    double rnorm = std::sqrt(h[0]);
    const double tol = std::max(o.rtol * bnorm, o.atol);
    int it = 0;
    bool conv = rnorm <= tol;
    // one PCG iteration: everything is enqueued on the stream with device-resident scalars, no host synchronisation
    auto iteration = [&](bool first) -> int {
        int r;
        if (pre != 0) {
            // z = M^-1 r ; rz' = r.z ; p = z + beta p
            if ((r = precond_apply(p, P, p->kr_r, p->kr_z))) return r;
            k_dot<<<go, kThreads, 0, st>>>(p->kr_r + p->own_off, p->kr_z + p->own_off, p->own_n, pa);
            p->launches++;
            if ((r = reduce_to(p, pa, nullptr, go, S_TMP0, 0))) return r;
            if ((r = scalar_op(p, first ? 3 : 2))) return r;
            k_cg_dir<<<g, kThreads, 0, st>>>(p->d_scalars, p->kr_r, nullptr, p->kr_z, p->kr_p, n, first);
            p->launches++;
        } else if (!first) {
            k_cg_dir<<<g, kThreads, 0, st>>>(p->d_scalars, p->kr_r, p->kr_dinv, nullptr, p->kr_p, n, 0);
            p->launches++;
        }
        // q = A p ; alpha = rz / p.q
        if ((r = outer(std::true_type{}, p->kr_p, p->kr_q))) return r;
        ++spmvs;
        if ((r = reduce_to(p, p->d_partials, nullptr, np, S_PQ, 0))) return r;
        if ((r = scalar_op(p, 0))) return r;
        // x += alpha p ; r -= alpha q
        if (pre == 0) {
            k_cg_update<<<g, kThreads, 0, st>>>(p->d_scalars, p->kr_p, p->kr_q, p->kr_dinv, x, p->kr_r, n, o0, o1, pa, pb);
            p->launches++;
            if ((r = reduce_to(p, pa, pb, g, S_TMP0, S_TMP1))) return r;
            if ((r = scalar_op(p, 1))) return r;
        } else {
            k_cg_update<<<g, kThreads, 0, st>>>(p->d_scalars, p->kr_p, p->kr_q, nullptr, x, p->kr_r, n, o0, o1, pa, pb);
            p->launches++;
            if ((r = reduce_to(p, pb, nullptr, g, S_RR, 0))) return r;
        }
        FEMO_CHECK_LAUNCH();
        return FEMO_OK;
    };
    // Launch-bound problems (every kernel of an iteration runs a few microseconds): the iteration body -- identical from
    // the second iteration on -- is captured into a CUDA graph once per solve and replayed (K9 of SURVEY.md section 8a).
    // One GPU only: the transport's kernels take a per-launch sequence number.
    cudaGraphExec_t gexec = nullptr;
    long long body_launches = 0;
    int body_spmvs = 0;
    bool graph_failed = false;
    while (!conv && it < o.max_it) {
        if (it >= 1 && use_graph && !graph_failed) {
            if (!gexec) {
                const long long l0 = total_launches(p);
                const int s0 = spmvs;
                cudaGraph_t graph = nullptr;
                bool ok = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
                int brc = FEMO_OK;
                if (ok) brc = iteration(false);
                cudaError_t ce = ok ? cudaStreamEndCapture(st, &graph) : cudaErrorUnknown;
                ok = ok && brc == FEMO_OK && ce == cudaSuccess && graph;
                if (ok) ok = cudaGraphInstantiate(&gexec, graph, 0) == cudaSuccess;
                if (graph) cudaGraphDestroy(graph);
                body_launches = total_launches(p) - l0;
                body_spmvs = spmvs - s0;
                if (!ok) {           // not capturable on this driver: fall back to plain launches for good
                    cudaGetLastError();
                    graph_failed = true;
                    gexec = nullptr;
                    p->launches -= body_launches;
                    spmvs = s0;
                    continue;
                }
                p->launches -= body_launches;     // the capture pass did not execute anything
                spmvs = s0;
            }
            FEMO_CUDA(cudaGraphLaunch(gexec, st));
            p->launches += body_launches;
            p->graph_replays++;
            spmvs += body_spmvs;
        } else if ((rc = iteration(it == 0))) {
            if (gexec) cudaGraphExecDestroy(gexec);
            return rc;
        }
        ++it;
        if (it % o.check_every == 0 || it >= o.max_it) {
            double rr;
            if ((rc = read_scalars(p, S_RR, 1, &rr))) {
                if (gexec) cudaGraphExecDestroy(gexec);
                return rc;
            }
            rnorm = std::sqrt(rr);
            if (!(rnorm == rnorm)) break;  // NaN
            conv = rnorm <= tol;
        }
    }
    if (gexec) cudaGraphExecDestroy(gexec);
    if ((rc = halo_nodes(p, x))) return rc;   // hand back a solution that is valid on the ghost rows too
    if (info) {
        info->iterations = it;
        info->converged = conv ? 1 : 0;
        info->rnorm = rnorm;
        info->bnorm = bnorm;
        info->spmv_count = spmvs;
    }
    return FEMO_OK;
}
