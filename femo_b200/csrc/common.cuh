// common.cuh -- shared device helpers and the problem object.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/femo_b200.h"
#include "layout.hpp"

namespace femo {

extern thread_local std::string g_err;
int set_err(int code, const std::string &msg);

#define FEMO_CUDA(call)                                                                      \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess)                                                              \
            return femo::set_err(FEMO_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)

#define FEMO_CHECK_LAUNCH() FEMO_CUDA(cudaGetLastError())

// Environment switches (debug / test toggles) are looked up once per C-ABI call, not per kernel launch: getenv is a
// linear scan of the environment and the solver enqueues a few thousand launches per step.
struct EnvFlags {
    bool no_bsr = false, no_dia = false, no_overlap = false, no_mgfused = false, no_mgsweep = false, no_lattice_asm = false, no_graph = false, force_graph = false;
    // A/B switches of the adjoint / set-up glue: FEMO_NO_TRANSPOSE_GATHER (transposed SpMV and adjoint DIA conversion through a permuted copy),
    // FEMO_MG_SETUP_SYNC_EACH (one host read per multigrid level), FEMO_NO_BAND_INVERSE (Gauss-Jordan sweeps every row)
    bool no_transpose_gather = false, mg_setup_sync_each = false, no_band_inverse = false;
    long long overlap_min_rows = 1 << 20, mgfused_max_rows = 20000, graph_max_rows = 1 << 20;
    long long mgfused_small_rows = 0;        // fused V-cycle ops up to this many rows run on ONE CTA (FEMO_MGFUSED_SMALL_ROWS); off:
                                             // measured slower (4096: 50.5 ms against 46.9 ms per step, profiles/r02_summary.md)
    long long mgfused_ctas = 0;              // CTAs of the cooperative coarse V-cycle (0: rows of its largest level / 512, FEMO_MGFUSED_CTAS)
};
extern EnvFlags g_env;
void refresh_env();

constexpr int kThreads = 256;
constexpr int kMaxPartials = 4096;   // upper bound on CTAs of any reducing kernel
constexpr int kMaxSlots = 12;

// device scalar slots (doubles) used by the Krylov / Newton drivers
enum Scalar { S_ALPHA = 0, S_BETA, S_RZ, S_RR, S_PQ, S_TMP0, S_TMP1, S_TMP2, S_BB, S_FLAG /* int flag raised by k_csr_to_dia */, S_GM = 16,
             S_MG = 96 /* multigrid set-up: S_TMP2..S_FLAG of each level, 3 slots per level */, S_COUNT = 128 };

// ---- reductions (deterministic: fixed assignment, fixed tree) ---------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// result valid in thread 0 of the block; safe to call repeatedly
__device__ __forceinline__ double block_sum(double v) {
    __shared__ double sh[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    v = warp_sum(v);
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.0;
    if (wid == 0) v = warp_sum(v);
    __syncthreads();
    return v;
}

// streaming loads for data touched once per kernel (matrix values / indices):
// keep L1/L2 for the gathered vector instead
__device__ __forceinline__ double ld_stream(const double *p) { return __ldcs(p); }
__device__ __forceinline__ int32_t ld_stream(const int32_t *p) { return __ldcs(p); }
__device__ __forceinline__ double f2d(float f) { return (double)f; }
__device__ __forceinline__ double ld_stream(const float *p) { return f2d(__ldcs(p)); }

// y-slab of a global lattice owned by this rank: global cell rows [crow0, crow0+ncrows) are local,
// local node row j is global row crow0 + j; node / cell rows [own0,own1) / [cown0,cown1) are owned
struct SlabInfo {
    bool active = false;
    int rank = 0, nranks = 1;
    int gny = 0, crow0 = 0, ncrows = 0;
    int own0 = 0, own1 = 0, cown0 = 0, cown1 = 0;
};

// General cell partition of an unstructured mesh (femo_b200/partition.py): this rank's problem lives on its LOCAL mesh --
// owned dofs first ([0, n_owned_dofs)), ghost dofs after them, owned cells first.  A halo exchange packs the owned values the
// neighbours hold as ghosts, all-gathers the (equal-sized, boundary-sized) send buffers of all ranks and scatters the
// entries this rank's ghosts need: one pack kernel, one collective of the existing transports, one unpack kernel.
struct GenPart {
    bool active = false;
    int64_t n_owned_dofs = 0, n_owned_cells = 0, blk = 0;     // blk: doubles per rank in the gathered buffer
    std::vector<int32_t> send_idx, ghost_src;                  // local dof -> send slot ; ghost dof k -> index into the gathered buffer
    int32_t *d_send_idx = nullptr, *d_ghost_src = nullptr;
    double *d_gather = nullptr;
};

struct DevPattern {
    int32_t *rowptr = nullptr, *col = nullptr, *gptr = nullptr, *gsrc = nullptr;
    int32_t *t_rowptr = nullptr, *t_col = nullptr, *t_perm = nullptr;
    uint8_t *bcflag = nullptr;
    int32_t *rb = nullptr, *t_rb = nullptr;  // SpMV row blocks
    int nrb = 0, t_nrb = 0;
    int32_t *b_rowptr = nullptr, *b_col = nullptr, *b_perm = nullptr, *b_rb = nullptr;   // 3x3 block view (layout.hpp)
    int nbrb = 0;
};
struct DevVecMap {
    int32_t *ptr = nullptr, *src = nullptr;
};

// Bump allocator over a caller-provided device buffer, in 256-byte slots.  Each arena is filled by one layout walk that
// runs in two modes.  An Arena without a buffer counts: take() only adds the rounded size to `used` and leaves its
// destination alone, so the same walk is the size query and writes nothing.  With a buffer the walk places and uploads:
// a take() that does not fit sets the sticky `failed` and hands out nullptr from then on, a failed copy is kept in
// `err`, and the caller checks both once at the end (check()).
struct Arena {
    char *base = nullptr;
    size_t cap = 0, used = 0;
    cudaStream_t stream = nullptr;   // the copies of put / put_soa
    bool failed = false;
    cudaError_t err = cudaSuccess;
    Arena() = default;
    Arena(void *b, size_t c, cudaStream_t s = nullptr) : base((char *)b), cap(c), stream(s) {}
    bool counting() const { return base == nullptr; }
    template <class T>
    void take(T *&dst, size_t count) {
        const size_t at = used;
        used += need(count, sizeof(T));
        if (counting()) return;
        failed |= used > cap;
        dst = failed ? nullptr : (T *)(base + at);
    }
    void copy(void *dst, const void *src, size_t bytes) {
        if (err == cudaSuccess) err = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    }
    // a placing walk succeeded: every copy was accepted and the layout took exactly the `counted` bytes of its count pass
    int check(size_t counted, const std::string &what) const {
        if (err != cudaSuccess) return set_err(FEMO_ECUDA, what + ": " + cudaGetErrorString(err));
        if (failed || used != counted)
            return set_err(FEMO_EINVAL, what + ": placed " + std::to_string(used) + " bytes, the size query counted " + std::to_string(counted));
        return FEMO_OK;
    }
    static size_t need(size_t count, size_t elem) { return (count * elem + 255) & ~size_t(255); }
};

// reserve a host array's slot (at least one element) and copy the array in
template <class T>
void put(Arena &A, T *&dst, const std::vector<T> &src) {
    A.take(dst, std::max<size_t>(1, src.size()));
    if (!A.counting() && !A.failed && !src.empty()) A.copy(dst, src.data(), src.size() * sizeof(T));
}
// the same for an array of structures with `ncomp` components per entity, placed as ncomp planes (SoA)
template <class T>
void put_soa(Arena &A, T *&dst, const std::vector<T> &aos, int ncomp) {
    A.take(dst, std::max<size_t>(1, aos.size()));
    if (A.counting() || A.failed) return;
    const size_t n = aos.size() / ncomp;
    std::vector<T> soa(aos.size());
    for (size_t e = 0; e < n; ++e)
        for (int a = 0; a < ncomp; ++a) soa[a * n + e] = aos[e * ncomp + a];
    if (!soa.empty()) A.copy(dst, soa.data(), soa.size() * sizeof(T));
    if (A.err == cudaSuccess) A.err = cudaStreamSynchronize(A.stream);   // soa goes out of scope
}

// DIA (diagonal) storage of a lattice operator: nd planes of np fp32 values, plane s holds a(i, i + off[s]);
// plane nd holds the Jacobi scaling (float)(1 / a_ii) used by every smoother step
constexpr int kDiaMax = 9;
struct DiaMat {
    const float *v = nullptr;
    int64_t np = 0, n = 0;
    int nd = 0, sdiag = 0;      // sdiag: the plane with off == 0
    int off[kDiaMax] = {0};
};

}  // namespace femo

struct femo_mesh {
    femo::Mesh m;
};

// device work vectors of one multigrid level (level 0 is the problem itself)
struct femo_mg_level {
    double *vals = nullptr;   // matrix values of this level (coarse levels own theirs)
    float *vals32 = nullptr;  // fp32 copy streamed by the V-cycle's SpMVs (8 instead of 12 bytes per entry)
    double *dinv = nullptr, *x = nullptr, *b = nullptr, *r = nullptr, *d = nullptr, *q = nullptr;
    double *u = nullptr;      // restricted state used to rediscretise the coarse Jacobian
    double *dense = nullptr, *dense_tmp = nullptr;  // coarsest level: explicit inverse
    double *m = nullptr;                            // restricted cell-wise input (SIMP density)
    double *ec = nullptr, *k0 = nullptr;            // hexahedral lattices: cell moduli rho^p and the unit-modulus 24x24
                                                    // element matrix of the level's (congruent) cells: matrix-free V-cycle
    double *fb = nullptr, *fx = nullptr;            // full-multigrid start: restricted right-hand side, nested iterate
    double lmax = 2.0;
    femo::DiaMat dia;                               // lattice stencil levels: the V-cycle streams DIA planes (stencil.cuh);
    bool dia_valid = false;                         // they alias the vals32 buffer
    double *dia64 = nullptr;                        // level 0: fp64 planes of the operator the Krylov recurrence applies
    bool dia64_valid = false;
};

namespace femo {
// ops of the cooperative coarse V-cycle kernel (mgfused.cuh)
enum MgOpType {
    MGO_PRE2 = 0,       // x = fused zero-guess degree-2 Chebyshev smoother of b
    MGO_RESID = 1,      // y = b - A x
    MGO_RESTRICT = 2,   // coarse b = P^T r          (nested 2:1 or general lattices)
    MGO_DENSE = 3,      // x = Inv b                 (coarsest level)
    MGO_PROLONG = 4,    // x += P xc
    MGO_CHEB0 = 5,      // r = b - A x ; d = c1 r / a_ii
    MGO_CHEBK = 6       // r' = r - A d ; x += d + c1 d + c2 r' / a_ii     (last step: r', d' not stored)
};

struct MgOp {
    int type = 0, nested = 0, n = 0, pad = 0;
    DiaMat A;
    const double *b = nullptr, *x = nullptr, *src = nullptr, *inv = nullptr;
    double *y = nullptr, *r = nullptr, *d = nullptr, *dst = nullptr;
    const uint8_t *mask_f = nullptr, *mask_c = nullptr;
    double c0 = 0.0, c1 = 0.0, c2 = 0.0;
    int fnx = 0, fny = 0, cnx = 0, cny = 0;     // fine / coarse lattice of a transfer
};

}  // namespace femo
// program of the cooperative coarse V-cycle kernel (mgfused.cuh): levels [k0, nlev-1] in one launch
struct MgFusedProg {
    bool valid = false, dirty = true;
    int k0 = 0, nops = 0, nlev = 0;
};

struct femo_amg;
struct femo_problem {
    femo::Mesh mesh;
    int family = 0;
    double params[32] = {0};
    femo::Space state, in[4], aux[4];
    int nin = 0, naux = 0, nout = 0;
    // integral blocks by mask: 1 = all cells, 2 = facets carrying facet integrals, 3 = both
    int res_mask = 1, jac_mask = 1, drdm_mask = 1;
    int out_mask[4] = {1, 1, 1, 1};        // blocks of output k's functional
    int out_du_mask[4] = {1, 1, 1, 1};     // blocks of d(output k)/d(state); 0 = identically zero
    int out_dm_mask[4] = {1, 1, 1, 1};     // same wrt input 0
    bool symmetric = true;
    bool lattice_fast = false;              // Jacobian rows assembled node-centrically on the lattice (lattice_asm.cuh)
    std::vector<int32_t> fb_cell, fb_local;   // the facets of block 2 (all exterior, or the tagged subset)
    std::vector<femo::IntegralBlock> blk[4];
    femo::Pattern pat[5];
    femo::VecMap vm_state[4], vm_in[4];     // vm_state indexed by block mask
    // Dirichlet data (host)
    bool has_bc = false;
    std::vector<uint8_t> bc_mark, bcflag;
    std::vector<double> bc_g, bc_diag;
    std::vector<int32_t> lift_rows;
    // device
    int device = -1;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;          // high-priority side stream: halo exchange + slab-boundary rows (overlap)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool uploaded = false;
    int num_sms = 148;
    double *d_coords = nullptr;
    int32_t *d_cellsT = nullptr, *d_fb_cell = nullptr, *d_fb_local = nullptr, *d_cell_tag = nullptr;
    // P2 spaces: edge opposite each local vertex (SoA), edge -> vertices, vertex -> incident edges (CSR)
    double *d_uex_tab = nullptr;   // angle-addition table of the analytic u_ex on uniform lattices (families 2, 9)
    int32_t *d_edgesT = nullptr, *d_edge_verts = nullptr, *d_vptr = nullptr, *d_vedge = nullptr;
    std::vector<int32_t> vptr, vedge;
    std::vector<double> h_uex_tab;   // host copy of the u_ex angle-addition table (copied to constant memory before its kernels)
    std::vector<double> h_k0;    // hexahedral lattices: host copy of the unit element matrix (kernel parameter of the matrix-free operator)
    femo::DevPattern dpat[5];
    femo::DevVecMap dvm_state[4], dvm_in[4];
    uint8_t *d_bc_mark = nullptr;
    double *d_bc_g = nullptr, *d_bc_diag = nullptr;
    int32_t *d_lift_rows = nullptr;
    // work
    double *d_scratch = nullptr, *d_partials = nullptr, *d_scalars = nullptr;
    double *kr_r = nullptr, *kr_p = nullptr, *kr_q = nullptr, *kr_dinv = nullptr, *kr_z = nullptr, *kr_w = nullptr;
    double *nt_b = nullptr, *nt_dx = nullptr, *nt_vals = nullptr, *nt_vals_bc = nullptr, *d_tvals = nullptr;
    double *h_pinned = nullptr;  // small pinned staging for scalars
    size_t scratch_len = 0, tvals_len = 0;
    // coefficients
    const double *coef[femo::kMaxSlots] = {nullptr};
    int64_t coefn[femo::kMaxSlots] = {0};
    // multi-GPU slab (inactive on one GPU); reductions run over the owned ranges only
    femo::SlabInfo slab;
    int64_t own_off = 0, own_n = 0;        // owned state dofs: [own_off, own_off + own_n)
    int64_t cown_off = 0, cown_n = 0;      // owned cells
    bool skip_next_halo = false; // set when the next halo_nodes() input provably has fresh ghost rows (consumed by that call)
    int face_mask = 0;           // hexahedral slabs: box faces tagged as traction facets
    int64_t fown_off = 0;        // first facet of block 2 whose cell is owned (facets are sorted by cell)
    bool replicated = false;               // multigrid level held identically by every rank
    bool mg_bc_dirty = false;              // replicated levels still need the gathered Dirichlet marks
    // geometric multigrid: coarse problems (owned), Jacobian-only layouts
    bool jac_only = false;
    std::vector<femo_problem *> mg;
    femo_mg_level mgl;
    femo_problem *parent = nullptr;
    double *kr_d = nullptr;
    double *d_bvals = nullptr;               // values re-laid out as 3x3 blocks for the Krylov recurrence (BSR-3 SpMV)
    double *d_dense = nullptr, *d_dense_tmp = nullptr;   // explicit inverse for small systems (precond 3)
    double *gm_basis = nullptr;                          // GMRES Krylov basis, (restart+1) vectors
    double *d_partials_big = nullptr, *wk_extra = nullptr; // multi-dot partials; spare N-vector
    int gm_restart = 0;
    // counters (bench: how many of our kernels were launched)
    MgFusedProg mgprog;
    femo::MgOp *d_mgops = nullptr;
    std::vector<femo::MgOp> h_mgops;
    femo::GenPart gpart;                     // unstructured partition (inactive on lattices / one GPU)
    struct femo_amg *amg = nullptr;          // smoothed-aggregation hierarchy (precond 4; amg.cuh), owned
    long long launches = 0;
    long long graph_replays = 0;             // PCG iterations replayed from a captured CUDA graph
    long long dia_count[4] = {0, 0, 0, 0};   // launches of the DIA operator kernel on this level, by mode
    long long dia64_count[2] = {0, 0};       // launches of the fp64 DIA SpMV on this level: with / without the fused dot
    long long sweep_count[2] = {0, 0};       // launches of the fused level sweeps (mgsweep.cuh) on this level: down / up
};
