/* femo_b200.h -- C ABI of libfemo_b200.so, the B200-native state/adjoint engine
 * that backs femo's FEA / CSDL operations.
 *
 * The reference (RuruX/femo) has no FFI: its hot path is a set of Python
 * one-liners that delegate to dolfinx 0.5.1 / PETSc / MUMPS.  Each entry point
 * below names the reference call it replaces (paths relative to the reference
 * root).  The Python host (femo_b200/fea, femo_b200/csdl_opt) binds these with
 * ctypes; INTEGRATION.md shows the stub a femo maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative FEMO_E* code on failure;
 *     femo_last_error() gives the message of the calling thread's last failure.
 *   - `d_*` pointers are DEVICE pointers owned by the caller (torch tensors on
 *     the Python side), `h_*` / unprefixed pointers are host memory.
 *   - all floating point is IEEE fp64, all indices int32 (dolfinx/PETSc default).
 *   - calls enqueue on the problem's stream; only functions that return a host
 *     scalar (or are documented to) synchronise.
 *   - there is NO CPU fallback: device entry points fail with FEMO_ENODEVICE
 *     when no CUDA device is present.
 */
#ifndef FEMO_B200_H
#define FEMO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEMO_OK 0
#define FEMO_EINVAL -1    /* bad argument                                    */
#define FEMO_ENODEVICE -2 /* CUDA device required but not present / not set  */
#define FEMO_ECUDA -3     /* CUDA runtime error                              */
#define FEMO_ESTATE -4    /* call order violated (e.g. not uploaded, no BC)  */
#define FEMO_ENOCONV -5   /* nonlinear solve did not converge (SNES semantics) */
#define FEMO_ELIMIT -6    /* problem exceeds int32 index range               */

typedef struct femo_mesh femo_mesh;
typedef struct femo_problem femo_problem;

/* ---- form families (SURVEY.md section 8a, "Form families") ---------------- */
#define FEMO_FAMILY_POISSON_P1 1   /* examples/poisson_opt/run_poisson_opt.py:32-38,74-76 */
#define FEMO_FAMILY_NLPOISSON_P1 2 /* examples/nonlinear_poisson_opt/run_nonlinear_poisson_opt.py:88-116,140-142 */
#define FEMO_FAMILY_EB_BEAM 3      /* examples/beam_thickness_opt/run_thickness_opt_cantilever_beam.py:71-85 */
#define FEMO_FAMILY_SIMP_Q1 4      /* examples/beam_topo_opt/run_topo_opt_cantilever_beam.py:62-86 */
#define FEMO_FAMILY_MOTOR_MM 6     /* examples/em_motor_opt/motor_pde.py:134-183,199-210 (hyperelastic mesh motion, Nitsche on dS/ds(1000)) */
#define FEMO_FAMILY_NLPOISSON_P2 9  /* config 2 with a quadratic Lagrange state (BASELINE.json configs[1] "P1/P2"; SURVEY 8d C2-P2); params alpha, beta */
#define FEMO_FAMILY_SIMP_HEX8 8    /* 3-D extension of examples/beam_topo_opt/run_topo_opt_cantilever_beam.py:62-86 on trilinear hexahedra (SURVEY 8d C4-3D); params nu, fx, fy, fz, penal */
#define FEMO_FAMILY_MOTOR_EM 7     /* examples/em_motor_opt/motor_pde.py:12-130,186-197 (nonlinear magnetostatics on a moving mesh) */
#define FEMO_FAMILY_RM_PLATE 10     /* Reissner-Mindlin plate (flat case of examples/test_shell_m3l/shell_pde.py:219-311): CG2 deflection x CG1^2
                                      rotations, reduced shear integration, penalty clamp; inputs thickness (CG1), load (CG1);
                                      outputs compliance, mass, elastic energy; params E, nu, pen, rho */
#define FEMO_FAMILY_MASS_P1 5      /* L2 projection, femo/fea/utils_dolfinx.py:549-583; params: target (0 CG1, 1 DG0),
                                      source (0 u_ex, 1 f_ex analytic; 2 DG0 input^power; 3 CG1 input), power */

/* matrix selector `which`: 0 = dR/du (N x N), 1+s = dR/dm_s (N x M_s) */

int femo_version(void);
const char *femo_last_error(void);
/* number of visible CUDA devices (0 on a CPU-only box; never fails) */
int femo_device_count(void);

/* ---- meshes: host only; replace dolfinx.mesh.create_* ---------------------
 * femo/fea/utils_dolfinx.py:136-153 (createUnitSquareMesh, createIntervalMesh,
 * createRectangleMesh).  Canonical lattice numbering, see DESIGN.md. */
int femo_mesh_create_unit_square(int nx, int ny, const double lo[2], const double hi[2], femo_mesh **out);
int femo_mesh_create_rectangle_quad(int nx, int ny, const double lo[2], const double hi[2], femo_mesh **out);
/* unstructured mesh from caller arrays: replaces import_mesh / XDMFFile.read_mesh (utils_dolfinx.py:69-123).
 * kind: 1 interval, 2 triangle, 3 quadrilateral, 4 hexahedron; cells hold vertex ids in basix order; coords is
 * (nverts, gdim).  No lattice structure is assumed: every family assembles on it, geometric multigrid is unavailable. */
int femo_mesh_create_from_arrays(int kind, int gdim, int64_t nverts, const double *coords, int64_t ncells, const int32_t *cells,
                                 femo_mesh **out);
/* hexahedral lattice on a box (dolfinx.mesh.create_box, CellType.hexahedron); vertex (ix,iy,iz) -> (iz*(ny+1)+iy)*(nx+1)+ix */
int femo_mesh_create_box_hex(int nx, int ny, int nz, const double lo[3], const double hi[3], femo_mesh **out);
int femo_mesh_create_interval(int n, double x0, double x1, femo_mesh **out);
/* synthetic stand-in for the motor meshes (git-LFS pointers in the reference): periodic polar lattice on
 * r0 <= r <= r1, node (ir, ith) -> ir*nth + ith */
int femo_mesh_create_annulus(int nr, int nth, double r0, double r1, femo_mesh **out);
/* sizes[0..5] = ncells, nverts, verts/cell, gdim, n exterior facets, mesh kind */
int femo_mesh_sizes(const femo_mesh *m, int64_t sizes[6]);
/* what: 0 coords (double nverts*gdim), 1 cells (int32 ncells*nvpc),
 *       2 exterior-facet cell (int32), 3 exterior-facet local index (int32) */
int femo_mesh_copy(const femo_mesh *m, int what, void *out);
void femo_mesh_destroy(femo_mesh *m);

/* ---- problem layout: host only ---------------------------------------------
 * Replaces dolfinx FunctionSpace/dofmap construction, create_matrix /
 * sparsity-pattern build (utils_dolfinx.py:390 and every assemble_matrix(form)
 * at :185,195,575) with a pattern and deterministic cell->nnz gather map built
 * ONCE (reference quirk B12).  The mesh is copied; it may be destroyed after. */
int femo_problem_create(const femo_mesh *m, int family, const double *params, int nparams, femo_problem **out);
/* Same, with the facets of a tagged measure ds(tag) (createCustomMeasure / meshtags,
 * utils_dolfinx.py:532-546; examples' ds_(100)): indices into the mesh's exterior-facet list. */
int femo_problem_create_tagged(const femo_mesh *m, int family, const double *params, int nparams,
                               const int32_t *facet_ids, int nfacets, femo_problem **out);
/* General form: explicit one-sided facets (cell, local facet) of the facet integrals (NULL = the family's
 * default) and a subdomain id per cell (meshtags of the cells, the dx(i) measures of motor_pde.py; may be NULL). */
int femo_problem_create_ex(const femo_mesh *m, int family, const double *params, int nparams, const int32_t *facet_cell,
                           const int32_t *facet_local, int nfacets, const int32_t *cell_tags, femo_problem **out);
/* change one family parameter after creation (e.g. the source scaling of the incremental EM solve,
 * run_motor_opt.py:231-250) */
int femo_problem_set_param(femo_problem *p, int index, double value);
void femo_problem_destroy(femo_problem *p);
/* sizes[0]=N (state dofs) [1]=n inputs [2]=n aux fields [3]=n outputs
 * [4..7]=M_s (input s dofs) [8..11]=aux field dofs [12]=n exterior facets */
int femo_problem_sizes(const femo_problem *p, int64_t sizes[16]);
/* info[0]=rows [1]=cols [2]=nnz [3]=number of element contributions */
int femo_problem_pattern_info(const femo_problem *p, int which, int64_t info[4]);
/* CSR pattern, column-sorted: rowptr (rows+1), col (nnz) */
int femo_problem_pattern(const femo_problem *p, int which, int32_t *rowptr, int32_t *col);
/* sorted segmented-reduction map: entry t sums scratch[src[ptr[t]..ptr[t+1])] */
int femo_problem_gather_map(const femo_problem *p, int which, int32_t *ptr, int32_t *src);
/* dirichletbc objects (fea_dolfinx.py:169-176): `dofs` is the concatenation of
 * nlists dof arrays, list_ptr (nlists+1) delimits them; a dof listed k times
 * gets diagonal k (dolfinx set_diagonal adds once per bc object).  g (N values,
 * or NULL for homogeneous) holds the prescribed values.  May be called before
 * or after femo_problem_upload (after: synchronises); nlists = 0 clears. */
int femo_problem_set_bc(femo_problem *p, const int32_t *dofs, const int32_t *list_ptr, int nlists, const double *g);

/* ---- multi-GPU: one process per GPU, y-slab partition, NCCL ------------------
 * What the reference only nominally gets from MPI/PETSc (SURVEY.md section 2.3): the lattice is cut
 * into nranks slabs of gny/nranks cell rows; each rank's local problem holds its rows plus one ghost
 * cell row below / one ghost node row above, so assembly of owned rows needs no communication;
 * SpMV inputs are halo-exchanged (ncclSend/Recv of whole rows) and Krylov / Newton scalars are
 * all-reduced, all on the problem's stream.
 * Rank 0 calls femo_comm_unique_id and ships the 128 bytes to the others (e.g. torch.distributed);
 * every rank then calls femo_comm_init once. */
int femo_comm_unique_id(char id[128]);
int femo_comm_init(const char id[128], int rank, int nranks, int device);
/* The engine's own transport over peer memory (csrc/link.cuh): halo exchanges, scalar all-reduces and level gathers are
 * single kernels that store into IPC-mapped windows of the peer GPUs (NVLink / NVSwitch) and spin on sequence flags.
 * femo_link_create allocates this rank's window (capacities in doubles; 0 = defaults) and returns its 64-byte IPC
 * handle; after an all-gather of the handles (any host channel) femo_link_open maps the peers and activates the
 * communicator.  Works for several ranks on ONE device as well.  femo_comm_init (NCCL) remains as an alternative. */
int femo_link_create(int device, size_t halo_cap, size_t gather_cap, char handle[64]);
int femo_link_open(const char *handles, int rank, int nranks);
int femo_link_error(void);
int femo_comm_finalize(void);
int femo_comm_stats(long long stats[2]);   /* [halo exchanges, all-reduces] issued so far */
/* Host only: the local problem of `rank` on the (nx x gny)-cell triangle lattice over [lo,hi]. */
int femo_problem_create_slab(int family, const double *params, int nparams, int nx, int gny, const double lo[2],
                             const double hi[2], int rank, int nranks, femo_problem **out);
/* z-slab of the (nx x ny x gnz)-cell hexahedral box for rank `rank` (SURVEY.md section 8e: cell partition with a one-cell
 * ghost layer; a z-plane of nodes is contiguous, so halo planes are sent in place).  face_mask bit l tags the exterior
 * facets with local facet id l (0 z=lo, 1 y=lo, 2 x=lo, 3 x=hi, 4 y=hi, 5 z=hi) as the traction measure ds(100). */
int femo_problem_create_slab_hex(int family, const double *params, int nparams, int nx, int ny, int gnz, const double lo[3],
                                 const double hi[3], int rank, int nranks, int face_mask, femo_problem **out);
/* info: active, rank, nranks, gny, first local cell row, local cell rows, owned node rows [own0,own1),
 * owned cell rows [cown0,cown1) (local indices), own_off, own_n (dofs), cown_off, cown_n (cells), nx, ny_local */
int femo_problem_slab_info(const femo_problem *p, int64_t info[16]);
/* the problem's own (local) mesh: same selectors as femo_mesh_sizes / femo_mesh_copy; for P2 states additionally
 * 4 = edge -> vertices (nedges,2) and 5 = cell -> edges (ncells,3), nedges = state dofs - vertices */
int femo_problem_mesh_sizes(const femo_problem *p, int64_t sizes[6]);
int femo_problem_mesh_copy(const femo_problem *p, int what, void *out);
/* Unstructured partitions (the engine-side counterpart of dolfinx's partitioner + index maps under MPI.COMM_WORLD,
 * utils_dolfinx.py:32,140-153; lists from femo_b200/partition.py).  The problem was created on this rank's LOCAL mesh:
 * owned nodes first, ghost nodes after them, owned cells first.  After femo_problem_upload: reductions and cell
 * functionals run over the owned ranges, every operator application refreshes the ghost dofs of its input (pack the
 * `n_send` owned nodes `send_nodes` the neighbours hold as ghosts -> all-gather of the ranks' send buffers, `blk_nodes`
 * nodes each -> ghost k reads gathered node `ghost_src_nodes[k]` = owner * blk_nodes + position), Krylov scalars are
 * all-reduced, and the AMG preconditioner (precond 4) smooths on the distributed level 0 (halo exchanges, global Chebyshev
 * bound) with a coarse correction local to the rank.
 * d_buf: caller-provided device buffer; call with d_buf = NULL to get the required size in *bytes. */
int femo_problem_set_partition(femo_problem *p, int64_t n_owned_nodes, int64_t n_owned_cells, int64_t blk_nodes, int64_t n_send,
                               const int32_t *send_nodes, int64_t n_ghost, const int32_t *ghost_src_nodes, void *d_buf,
                               int64_t *bytes);
/* refresh ghost rows of a device vector: kind 0 = state-space (nodes), 1 = cell-wise input */
int femo_halo_exchange(femo_problem *p, double *d_v, int kind);

/* Build the geometric-multigrid hierarchy used by Krylov precond = 2 (coarse
 * lattices, Jacobian-only layouts).  Host only; must precede upload.  Scalar P1
 * states on lattice triangle meshes. */
int femo_problem_enable_multigrid(femo_problem *p);
int femo_problem_mg_levels(const femo_problem *p);

/* ---- device residency ------------------------------------------------------
 * Bytes the caller must provide: static (maps, patterns) and work (scratch,
 * Krylov vectors), for the problem and its multigrid levels.  Both figures are
 * exact: the size query counts the same layout that upload places, and upload
 * fails if the two ever differ.  Host only; no device is needed.  Upload copies
 * the layout into d_static.  stream is a cudaStream_t (NULL = legacy default
 * stream). */
int femo_problem_device_bytes(const femo_problem *p, size_t *static_bytes, size_t *work_bytes);
int femo_problem_upload(femo_problem *p, int device, void *stream, void *d_static, size_t static_bytes,
                        void *d_work, size_t work_bytes);
/* coefficient slots: 0 = state, 1..nin = inputs, then aux fields.  Borrowed
 * device pointer, read at every assemble (update()/setFuncArray,
 * utils_dolfinx.py:161-167,300-311). */
int femo_set_coefficient(femo_problem *p, int slot, const double *d_values, int64_t n);

/* number of kernels this problem has launched so far (bench.py's gpu_launches) */
int femo_problem_launch_count(const femo_problem *p, long long *count);
/* PCG iterations replayed from a captured CUDA graph so far (launch-bound problems, csrc/krylov.cuh) */
int femo_problem_graph_replays(const femo_problem *p, long long *count);

/* ---- assembly --------------------------------------------------------------*/
/* assembleVector(residual_form): no BC applied (utils_dolfinx.py:175-179,
 * state_model.py:85). */
int femo_assemble_residual(femo_problem *p, double *d_out);
/* assembleMatrix(dR_du) and assembleSystem(dR_du, res, bcs) in ONE pass
 * (utils_dolfinx.py:181-202; state_model.py:132,149-151; quirk B8): writes the
 * un-BC'd values to d_vals and/or the BC'd copy (rows+cols zeroed, diagonal =
 * bc multiplicity) to d_vals_bc; either may be NULL. */
int femo_assemble_jacobian(femo_problem *p, double *d_vals, double *d_vals_bc);
/* assembleMatrix(derivative(res, m_s)), never BC'd (state_model.py:136-146). */
int femo_assemble_dRdm(femo_problem *p, int slot, double *d_vals);
/* NonlinearProblem.F / NonlinearSNESProblem.F (utils_dolfinx.py:352-367):
 * b = R(x) - scale*A(:,bc)(g-x), b[bc] = scale*(g-x) with scale=-1; d_vals is
 * the un-BC'd Jacobian at the same state. */
int femo_newton_rhs(femo_problem *p, const double *d_vals, double *d_b);
/* right-hand side of assembleSystem (utils_dolfinx.py:197-201): apply_lifting with
 * x0 = None, scale = 1, then set_bc:  b = R - A(:,bc) g, b[bc] = g. */
int femo_assemble_system_rhs(femo_problem *p, const double *d_vals, double *d_b);
/* assemble(form, dim=0) (utils_dolfinx.py:169-173,204-213; output_model.py:69-75).
 * Synchronises. */
int femo_assemble_output(femo_problem *p, int out_id, double *h_value);
/* assemble(derivative(form, arg), dim=1) (output_model.py:77-87); slot as in
 * femo_set_coefficient (0 = wrt state). */
int femo_assemble_output_grad(femo_problem *p, int out_id, int slot, double *d_out);
/* J and dJ/du in one quadrature pass (output_model.py:69-87 call both on the same state); synchronises. */
int femo_assemble_output_and_grad(femo_problem *p, int out_id, double *h_value, double *d_dJdu);

/* ---- linear algebra --------------------------------------------------------*/
/* computeMatVecProductFwd / Bwd (utils_dolfinx.py:256-264,275-287):
 * y = A x (transpose=0) or y = A^T x (transpose=1). */
int femo_spmv(femo_problem *p, int which, const double *d_vals, const double *d_x, double *d_y, int transpose);

/* The same product with the values re-laid out as 3x3 blocks (BSR-3: one column index per nine values, 8.44 instead of
 * 12 bytes per entry; what the CG recurrence streams for vector states in 3-D).  convert != 0 refreshes the block
 * copy from d_vals first. */
int femo_spmv_bsr3(femo_problem *p, const double *d_vals, const double *d_x, double *d_y, int convert);

/* y += a x on the problem's stream (the d_inputs accumulation of
 * compute_jacvec_product, state_model.py:180-199, kept on the device). */
int femo_axpy(femo_problem *p, double a, const double *d_x, double *d_y, int64_t n);

/* Cone density filter of examples/beam_topo_opt/pre_processor/general_filter_model.py:33-90 on the lattice of
 * cell centres (nx x ny cells of size dx x dy, cell id = j*nx + i): out = W in, W_ij = (R-d_ij)/sum_k(R-d_ik)
 * for d <= R, or out = W^T in (the constant Jacobian's transpose action).  d_den: nx*ny doubles of scratch. */
int femo_filter_apply(int device, void *stream, int nx, int ny, double dx, double dy, double radius,
                      const double *d_in, double *d_out, double *d_den, int transpose);
/* The same filter on a 3-D lattice of cell centres (nx x ny x nz, cell id = (k*ny + j)*nx + i): the pre-processor of
 * the 16.8M-cell cantilever (SURVEY.md section 8f rank 1); d_den: nx*ny*nz doubles of scratch. */
int femo_filter_apply3(int device, void *stream, int nx, int ny, int nz, double dx, double dy, double dz, double radius,
                       const double *d_in, double *d_out, double *d_den, int transpose);
/* out = a * num / den (Vec.pointwiseDivide of the lumped projection, utils_dolfinx.py:566-569) */
int femo_pointwise_divide(femo_problem *p, double a, const double *d_num, const double *d_den, double *d_out, int64_t n);

/* Host-side bulk helpers for the API boundary (no device code): the femo callbacks assign and accumulate dense fp64
 * numpy vectors (state_model.py:75-200); these run dst = alpha*src, dst += alpha*src and dst = value on all host cores. */
void femo_host_scaled_copy(double *dst, const double *src, int64_t n, double alpha);
void femo_host_axpy(double *dst, const double *src, int64_t n, double alpha);
void femo_host_fill(double *dst, int64_t n, double value);

typedef struct femo_krylov_opts {
    double rtol;      /* ||r|| <= rtol*||b||   */
    double atol;      /* or ||r|| <= atol      */
    int max_it;
    int precond;      /* 0 Jacobi, 1 Chebyshev polynomial of the Jacobi-scaled operator (cheb_degree, cheb_ratio),
                         2 geometric multigrid V-cycle (Chebyshev-Jacobi smoothing),
                         3 explicit dense inverse (N <= 512; the direct-solve analogue),
                         4 smoothed-aggregation algebraic multigrid V-cycle (femo_amg_symbolic + femo_amg_attach first;
                           meshes without a lattice hierarchy) */
    int cheb_degree;  /* smoother degree of the V-cycle, precond 2 and 4 (default 2) */
    int method;       /* 0 CG, 1 restarted GMRES (right-preconditioned, CGS2; non-symmetric Jacobians) */
    int restart;      /* GMRES restart; with precond 2: 1 disables the full-multigrid start */
    int check_every;  /* residual-norm host check period (>=1) */
    double cheb_ratio; /* smoother targets [lmax/ratio, lmax] of D^-1 A (default 8) */
    int mg_precision;  /* precond 2: 0 = the V-cycle streams fp32 copies of the level matrices (vectors, the outer
                          Krylov recurrence and every residual stay fp64), 1 = fp64 values throughout */
    double forcing;    /* femo_newton_solve only: > 0 = inexact Newton, the relative tolerance of each linear solve follows
                          Eisenstat-Walker's choice 2 between rtol and this eta_max (0: every solve to rtol) */
} femo_krylov_opts;

typedef struct femo_krylov_info {
    int iterations;
    int converged;
    double rnorm, bnorm;
    int spmv_count;
} femo_krylov_info;

/* Replaces KSP preonly + LU(MUMPS): solveKSP_mumps / setUpKSP_MUMPS and the
 * explicit transpose(A) (utils_dolfinx.py:241-245,476-512; fea_dolfinx.py:
 * 192-222).  Solves A x = b or A^T x = b on the dR/du pattern.  x is the
 * initial guess on entry for precond 0/1/3; with the multigrid preconditioner
 * (precond 2) the full-multigrid iterate REPLACES the caller's x unless
 * opts.restart == 1 (then x is honoured as x0).  Synchronises. */
int femo_linear_solve(femo_problem *p, const double *d_vals, const double *d_b, double *d_x, int transpose,
                      const femo_krylov_opts *opts, femo_krylov_info *info);

/* ---- algebraic multigrid for problems without a lattice hierarchy (unstructured meshes, the motor annulus) -------
 * The reference factorises every Jacobian with MUMPS (utils_dolfinx.py:405-408,476-512); precond 4 replaces that by a
 * smoothed-aggregation V-cycle.  femo_amg_symbolic (host only, once per pattern): strength graph, aggregates, the
 * patterns of P, R = P^T, A P, P^T A P on every level and the index lists of the numeric phase.  h_vals: host copy of
 * a (BC'd) Jacobian on the state pattern for the strength-of-connection test, or NULL (every connection strong).
 * Dirichlet rows (femo_problem_set_bc) are left out of the aggregates.  info[0] levels, info[1] bytes of device memory
 * femo_amg_attach needs (exact: the layout attach places, counted), info[2] sum of nnz over the levels, info[3] dofs of
 * the coarsest level.  femo_amg_attach uploads the lists into the caller's buffer (a torch tensor, like the problem
 * arenas).  The numeric phase (diagonals, Gershgorin bounds, prolongator values, Galerkin products: sorted segmented
 * reductions, no atomics) runs on the device at the start of every precond-4 solve; femo_amg_numeric runs it alone. */
typedef struct femo_amg_opts {
    double theta;        /* strength threshold |a_ij| >= theta sqrt(a_ii a_jj) on level 0 (default 0.08; < 0 keeps it) */
    double theta_decay;  /* factor per coarser level (default 0.5) */
    int max_levels;      /* default 10 */
    int coarse_size;     /* stop coarsening at this many dofs (default 200, dense inverse up to 512) */
    int block;           /* dofs per node (default: the state space's block size) */
    int omega_scale_set; /* nonzero: use omega_scale below */
    double omega_scale;  /* prolongator smoothing P = (I - omega_scale * 4/(3 lmax) D^-1 A) T (default 1; 0 = plain aggregation) */
} femo_amg_opts;
int femo_amg_symbolic(femo_problem *p, const double *h_vals, const femo_amg_opts *opts, int64_t info[4]);
int femo_amg_attach(femo_problem *p, void *d_arena, int64_t bytes);
int femo_amg_numeric(femo_problem *p, const double *d_vals);
/* Introspection for the tests: sizes (n, nnz, coarse n, nnz(P), nnz(AP), pairs of A P, pairs of P^T A P, sources of P) and
 * Gershgorin bounds (host phase, device phase); the integer lists (which: 0 rowptr, 1 col, 2 aggregate of each dof,
 * 3 p_rowptr, 4 p_col, 5 pp_ptr, 6 pp_src, 7 r_rowptr, 8 r_col, 9 r_perm, 10 ap_rowptr, 11 ap_col, 12 ap_ptr, 13 ap_ia,
 * 14 ap_ib, 15 ac_ptr, 16 ac_ia, 17 ac_ib); the values (which: 0 operator, 1 prolongator, 2 A P, 3 inverse diagonal) of
 * the host numeric phase or, from_device = 1, of the last device numeric phase. */
int femo_amg_level_info(const femo_problem *p, int level, int64_t info[8], double dinfo[2]);
int femo_amg_level_array(const femo_problem *p, int level, int which, int32_t *h_out, int64_t cap);
int femo_amg_level_values(femo_problem *p, int level, int which, int from_device, double *h_out, int64_t cap);

/* Measurement hook for bench.py's roofline (no reference counterpart): ONE launch of a fine-level operator kernel of
 * the last precond=2 solve on the solver's own work vectors.  mode 0 residual, 1 / 2 Chebyshev steps, 3 fused
 * zero-guess pre-smoother (fp32 DIA planes of the V-cycle); 4 / 5 the fp64 DIA SpMV of the CG recurrence with / without
 * the fused dot product; 6 / 7 the down / up level sweep of the V-cycle (pre-smoother + residual + restriction /
 * prolongation + post-smoother in one kernel each; FEMO_ESTATE when the fine level does not take the sweeps).
 * info[0] receives the algorithmic bytes of that launch (DESIGN.md section 3), info[1] the fine-level launches of that
 * mode so far. */
int femo_vcycle_op_probe(femo_problem *p, int mode, int64_t info[2]);

typedef struct femo_newton_opts {
    int kind;        /* 0 = dolfinx NewtonSolver (utils_dolfinx.py:419-449), 1 = PETSc SNES newtonls (:376-416) */
    double atol, rtol, stol;
    int max_it;
    femo_krylov_opts krylov;
} femo_newton_opts;

typedef struct femo_newton_info {
    int iterations;
    int converged;    /* SNES: 1 abs, 2 rel, 3 stol; Newton: 1 if tolerance met */
    double fnorm0, fnorm;
    int krylov_iterations; /* summed over Newton steps */
    int spmv_count;
} femo_newton_info;

/* FEA.solve -> solveNonlinear (fea_dolfinx.py:178-189, utils_dolfinx.py:319-333).
 * The state is coefficient slot 0 (updated in place).  SNES kind returns
 * FEMO_ENOCONV at max_it (error_on_nonconvergence, :399); Newton kind never
 * fails (quirk B1).  Synchronises. */
int femo_newton_solve(femo_problem *p, const femo_newton_opts *opts, femo_newton_info *info);

#ifdef __cplusplus
}
#endif
#endif /* FEMO_B200_H */
