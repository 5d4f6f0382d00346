// mgfused.cuh -- the coarse part of the V-cycle as ONE cooperative kernel.
//
// Below a few hundred thousand dofs a multigrid level is launch-latency bound: every smoother step, transfer and
// residual is a 3-6 us kernel that moves a few MB out of L2.  The levels [k0, coarsest] of a DIA hierarchy are
// therefore executed by a single persistent cooperative kernel (one CTA per SM) that interprets a small op list built
// at set-up time -- fused pre-smoother, residual, restriction, ..., dense coarsest solve, prolongation, two Chebyshev
// steps -- with a grid-wide barrier between dependent ops instead of a kernel boundary.  Same arithmetic, same order
// per row as the per-level kernels of stencil.cuh / multigrid.cuh (the row bodies are shared), so iterates agree.
//
// Included by engine.cu after stencil.cuh and multigrid.cuh's kernels.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace femo {

constexpr int kMgFusedMaxOps = 96;
constexpr int kMgFusedThreads = 512;

__device__ __forceinline__ double dia7_row(const DiaMat &A, int64_t i, const double *x, float &ad, double &xi) {
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < 7; ++s) {
        const float a = A.v[(int64_t)s * A.np + i];
        const int64_t j = i + A.off[s];
        const double v = (j >= 0 && j < A.n) ? __ldcg(x + j) : 0.0;
        if (s == 3) { ad = a; xi = v; }
        acc = fma((double)a, v, acc);
    }
    return acc;
}

// one op over the whole grid (grid-stride); vectors written by earlier ops of the same kernel on other SMs are read
// with ld.global.cg (L2 only: neither the non-coherent path nor a stale L1 line can be hit)
__device__ void mg_run_op(const MgOp &o, int64_t tid, int64_t nth) {
    switch (o.type) {
        case MGO_PRE2: {
            const DiaMat &A = o.A;
            const float *dg = A.v + 7 * A.np;      // dinv plane
            for (int64_t i = tid; i < A.n; i += nth) {
                double acc = 0.0, d0i = 0.0;
                float ad = 0.0f;
#pragma unroll
                for (int s = 0; s < 7; ++s) {
                    const float a = A.v[(int64_t)s * A.np + i];
                    const int64_t j = i + A.off[s];
                    double v = 0.0;
                    if (j >= 0 && j < A.n) v = o.c0 * (double)dg[j] * __ldcg(o.b + j);
                    if (s == 3) { ad = a; d0i = v; }
                    acc = fma((double)a, v, acc);
                }
                const double r = __ldcg(o.b + i) - acc;
                o.y[i] = d0i + o.c1 * d0i + o.c2 * (double)dg[i] * r;
            }
            break;
        }
        case MGO_RESID: {
            for (int64_t i = tid; i < o.A.n; i += nth) {
                float ad;
                double xi;
                const double acc = dia7_row(o.A, i, o.x, ad, xi);
                o.y[i] = __ldcg(o.b + i) - acc;
            }
            break;
        }
        case MGO_CHEB0: {
            for (int64_t i = tid; i < o.A.n; i += nth) {
                float ad;
                double xi;
                const double acc = dia7_row(o.A, i, o.x, ad, xi);
                const double r = __ldcg(o.b + i) - acc;
                o.r[i] = r;
                o.d[i] = o.c1 * (double)o.A.v[7 * o.A.np + i] * r;
            }
            break;
        }
        case MGO_CHEBK: {
            for (int64_t i = tid; i < o.A.n; i += nth) {
                float ad;
                double di;
                const double acc = dia7_row(o.A, i, o.x /* = d */, ad, di);
                const double r = __ldcg(o.b + i) /* = r */ - acc;
                const double dn = o.c1 * di + o.c2 * (double)o.A.v[7 * o.A.np + i] * r;
                o.y[i] = __ldcg(o.y + i) + di + dn;
            }
            break;
        }
        case MGO_RESTRICT: {
            const int64_t nc = (int64_t)(o.cnx + 1) * (o.cny + 1);
            if (o.nested) {
                const LatD f{o.fnx, o.fny + 1, 0}, c{o.cnx, o.cny + 1, 0};
                for (int64_t i = tid; i < nc; i += nth) restrict_nested_at<true>(f, c, o.src, o.dst, o.mask_f, o.mask_c, i);
            } else {
                const Lattice f{o.fnx, o.fny}, c{o.cnx, o.cny};
                for (int64_t i = tid; i < nc; i += nth) lattice_restrict_at<true>(f, c, 1, 0, o.src, o.dst, o.mask_f, o.mask_c, i);
            }
            break;
        }
        case MGO_PROLONG: {
            const int64_t nf = (int64_t)(o.fnx + 1) * (o.fny + 1);
            if (o.nested) {
                const LatD f{o.fnx, o.fny + 1, 0}, c{o.cnx, o.cny + 1, 0};
                for (int64_t i = tid; i < nf; i += nth) prolong_nested_at<true>(f, c, o.src, o.dst, o.mask_f, i);
            } else {
                const Lattice f{o.fnx, o.fny}, c{o.cnx, o.cny};
                for (int64_t i = tid; i < nf; i += nth) lattice_interp_at<true, true>(c, f, 1, 0, o.src, o.dst, o.mask_f, i);
            }
            break;
        }
        case MGO_DENSE: {
            const int n = o.n;
            const int64_t warp = tid >> 5, nwarps = nth >> 5;
            const int lane = (int)(tid & 31);
            for (int64_t row = warp; row < n; row += nwarps) {
                double acc = 0.0;
                for (int j = lane; j < n; j += 32) acc += o.inv[row * n + j] * __ldcg(o.b + j);
                acc = warp_sum(acc);
                if (lane == 0) o.y[row] = acc;
            }
            break;
        }
    }
}

// b0 / x0: right-hand side and solution of the first level of the program (they change from call to call);
// ops that refer to them carry the sentinel pointers (1 = b0, 2 = x0)
// work items of an op (rows it writes)
__device__ __forceinline__ int64_t mg_op_work(const MgOp &o) {
    switch (o.type) {
        case MGO_RESTRICT: return (int64_t)(o.cnx + 1) * (o.cny + 1);
        case MGO_PROLONG: return (int64_t)(o.fnx + 1) * (o.fny + 1);
        case MGO_DENSE: return o.n;
        default: return o.A.n;
    }
}

// Ops that write at most `small_rows` rows (the bottom of the hierarchy: a few thousand rows and the dense coarsest solve)
// are executed by CTA 0 alone, ordered by __syncthreads(); the other CTAs skip them and wait at the next grid-wide
// barrier.  A run of small ops therefore costs two grid barriers (entering and leaving it) instead of one per op.
// Measured on the B200 with small_rows = 4096 (levels of 3969 and 1024 rows + the dense solve on one CTA): 50.5 ms per
// step against 46.9 ms with every op grid-wide -- one SM's L2 latency chain is slower than 13 grid barriers -- so the
// default is 0 (off); FEMO_MGFUSED_SMALL_ROWS enables it.
__global__ void __launch_bounds__(kMgFusedThreads)
    k_mg_fused(const MgOp *__restrict__ ops, int nops, const double *b0, double *x0, int small_rows) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    for (int k = 0; k < nops; ++k) {
        MgOp op = ops[k];                       // uniform read-only loads (the list is constant during the kernel)
        if (op.b == (const double *)1) op.b = b0;
        if (op.x == (const double *)2) op.x = x0;
        if (op.y == (double *)2) op.y = x0;
        if (op.dst == (double *)2) op.dst = x0;
        const bool small = mg_op_work(op) <= small_rows;
        if (!small) mg_run_op(op, tid, nth);
        else if (blockIdx.x == 0) mg_run_op(op, threadIdx.x, blockDim.x);
        if (k + 1 < nops) {
            if (small && mg_op_work(ops[k + 1]) <= small_rows) {
                if (blockIdx.x == 0) __syncthreads();       // CTA 0 continues alone (block-uniform branch)
            } else {
                grid.sync();
            }
        }
    }
}

}  // namespace femo

using namespace femo;

// ---- host side -----------------------------------------------------------------------------------------------
// levels up to this many rows join the cooperative kernel (FEMO_MGFUSED_MAX_ROWS overrides; measured trade-off in DESIGN.md)
static int64_t mgfused_max_rows() { return g_env.mgfused_max_rows; }

// (re)build the op list for levels [k0, coarsest] with the smoother parameters of `mp`; called lazily by the first
// V-cycle after a set-up (the Chebyshev coefficients depend on the level bounds lmax computed there)
static int mgfused_build(femo_problem *root, const MgParams &mp) {
    MgFusedProg &P = root->mgprog;
    P.valid = false;
    P.dirty = false;
    const int nlev = (int)root->mg.size() + 1;
    if (nlev < 2 || mp.degree != 2 || !mp.fp32 || !root->d_mgops || g_env.no_mgfused) return FEMO_OK;
    int coop = 0;
    FEMO_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, root->device));
    if (!coop) return FEMO_OK;
    if (!mg_level(root, nlev - 1)->mgl.dense) return FEMO_OK;
    int k0 = nlev - 1;
    while (k0 > 0) {
        femo_problem *L = mg_level(root, k0 - 1);
        if (level_op(L, mp.fp32) != LevelOp::DIA || L->slab.active || L->state.ndofs > mgfused_max_rows()) break;
        --k0;
    }
    if (k0 >= nlev - 1) return FEMO_OK;
    if (6 * (nlev - 1 - k0) + 1 > kMgFusedMaxOps) return FEMO_OK;
    std::vector<MgOp> &ops = root->h_mgops;
    ops.clear();
    auto bptr = [&](int lv) { return lv == k0 ? (const double *)1 : (const double *)mg_level(root, lv)->mgl.b; };
    auto xptr = [&](int lv) { return lv == k0 ? (double *)2 : mg_level(root, lv)->mgl.x; };
    auto coef = [&](femo_problem *L) {       // degree 2: the PRE2 step and the CHEB0 / CHEBK pair share c0, c1, c2
        ChebPoly c(L->mgl.lmax, mp.ratio);
        c.next();
        return c;
    };
    auto transfer = [&](MgOp &o, femo_problem *F, femo_problem *C) {
        o.nested = nested_pair(F, C) ? 1 : 0;
        o.fnx = F->mesh.n[0]; o.fny = F->mesh.n[1]; o.cnx = C->mesh.n[0]; o.cny = C->mesh.n[1];
        o.mask_f = F->has_bc ? F->d_bc_mark : nullptr;
        o.mask_c = C->has_bc ? C->d_bc_mark : nullptr;
    };
    for (int lv = k0; lv < nlev - 1; ++lv) {        // down sweep
        femo_problem *L = mg_level(root, lv), *C = mg_level(root, lv + 1);
        const ChebPoly c = coef(L);
        MgOp o;
        o.type = MGO_PRE2; o.A = L->mgl.dia; o.b = bptr(lv); o.y = xptr(lv); o.c0 = c.c0; o.c1 = c.c1; o.c2 = c.c2;
        ops.push_back(o);
        o = MgOp();
        o.type = MGO_RESID; o.A = L->mgl.dia; o.x = xptr(lv); o.b = bptr(lv); o.y = L->mgl.r;
        ops.push_back(o);
        o = MgOp();
        o.type = MGO_RESTRICT; o.src = L->mgl.r; o.dst = C->mgl.b;
        transfer(o, L, C);
        ops.push_back(o);
    }
    {
        femo_problem *L = mg_level(root, nlev - 1);
        MgOp o;
        o.type = MGO_DENSE; o.n = (int)L->state.ndofs; o.inv = L->mgl.dense; o.b = L->mgl.b; o.y = L->mgl.x;
        ops.push_back(o);
    }
    for (int lv = nlev - 2; lv >= k0; --lv) {       // up sweep
        femo_problem *L = mg_level(root, lv), *C = mg_level(root, lv + 1);
        const ChebPoly c = coef(L);
        MgOp o;
        o.type = MGO_PROLONG; o.src = C->mgl.x; o.dst = xptr(lv);
        transfer(o, L, C);
        ops.push_back(o);
        o = MgOp();
        o.type = MGO_CHEB0; o.A = L->mgl.dia; o.x = xptr(lv); o.b = bptr(lv); o.r = L->mgl.r; o.d = L->mgl.d; o.c1 = c.c0;
        ops.push_back(o);
        o = MgOp();
        o.type = MGO_CHEBK; o.A = L->mgl.dia; o.x = L->mgl.d; o.b = L->mgl.r; o.y = xptr(lv); o.c1 = c.c1; o.c2 = c.c2;
        ops.push_back(o);
    }
    FEMO_CUDA(cudaMemcpyAsync(root->d_mgops, ops.data(), ops.size() * sizeof(MgOp), cudaMemcpyHostToDevice, root->stream));
    P.k0 = k0;
    P.nops = (int)ops.size();
    P.nlev = nlev;
    P.valid = true;
    return FEMO_OK;
}

// run the V-cycle of level lv >= k0 (b, x as mg_vcycle) in one cooperative launch; *done = false when this
// (level, b, x) combination is not covered by the program and the caller must take the per-kernel path
static int mgfused_vcycle(femo_problem *root, int lv, const double *b, double *x, const MgParams &mp, bool *done) {
    *done = false;
    MgFusedProg &P = root->mgprog;
    int rc;
    if (P.dirty && (rc = mgfused_build(root, mp))) return rc;
    if (!P.valid || lv < P.k0 || lv >= P.nlev - 1 || mp.degree != 2 || !mp.fp32) return FEMO_OK;
    {   // inside a stream capture (CUDA-graph replay of the PCG iteration) the per-level kernels are recorded instead:
        // a cooperative launch is not capturable, and a graph has no launch overhead to save anyway
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(root->stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) return FEMO_OK;
    }
    femo_problem *L = mg_level(root, lv);
    // ops of the first level of the (sub-)program take b / x from the launch; deeper starts must match the level's own vectors
    int first = 3 * (lv - P.k0), count = P.nops - 6 * (lv - P.k0);
    const double *b0 = b;
    double *x0 = x;
    if (lv > P.k0 && (b != L->mgl.b || x != L->mgl.x)) return FEMO_OK;
    const MgOp *ops = root->d_mgops + first;
    int small_rows = (int)g_env.mgfused_small_rows;
    void *args[] = {(void *)&ops, (void *)&count, (void *)&b0, (void *)&x0, (void *)&small_rows};
    // grid: one thread per row of the largest fused level is enough (a grid-wide barrier costs more the more CTAs arrive);
    // never more than one CTA per SM (co-residency of the cooperative launch)
    int64_t ctas = g_env.mgfused_ctas > 0 ? g_env.mgfused_ctas : (mg_level(root, P.k0)->state.ndofs + kMgFusedThreads - 1) / kMgFusedThreads;
    ctas = std::max<int64_t>(8, std::min<int64_t>(ctas, root->num_sms));
    FEMO_CUDA(cudaLaunchCooperativeKernel((const void *)k_mg_fused, dim3((unsigned)ctas), dim3(kMgFusedThreads), args, 0, root->stream));
    L->launches++;
    *done = true;
    return FEMO_OK;
}
