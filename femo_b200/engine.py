"""Object wrappers over the C ABI.  torch tensors are used ONLY as device
buffers (allocation, H2D/D2H copies, stream handles); every computation is a
libfemo_b200 call.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import lib, check, KrylovOpts, KrylovInfo, NewtonOpts, NewtonInfo

_DP_T = C.POINTER(C.c_double)
_I32P_T = C.POINTER(C.c_int32)
FAMILY_POISSON_P1 = 1
FAMILY_NLPOISSON_P1 = 2
FAMILY_EB_BEAM = 3
FAMILY_SIMP_Q1 = 4
FAMILY_MASS_P1 = 5
FAMILY_MOTOR_MM = 6
FAMILY_MOTOR_EM = 7
FAMILY_SIMP_HEX8 = 8
FAMILY_NLPOISSON_P2 = 9
FAMILY_RM_PLATE = 10


def device_count():
    return lib.femo_device_count()


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class EngineMesh:
    """Host-side structured mesh (replaces dolfinx.mesh.create_*)."""

    def __init__(self, handle):
        self._h = handle
        s = (C.c_int64 * 6)()
        check(lib.femo_mesh_sizes(self._h, s))
        self.ncells, self.nverts, self.nvpc, self.gdim, self.nbfacets, self.kind = [int(v) for v in s]

    @classmethod
    def unit_square(cls, nx, ny=None, lo=(0.0, 0.0), hi=(1.0, 1.0)):
        ny = nx if ny is None else ny
        h = C.c_void_p()
        check(lib.femo_mesh_create_unit_square(int(nx), int(ny), (C.c_double * 2)(*lo), (C.c_double * 2)(*hi), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = (nx, ny), tuple(lo), tuple(hi)
        return m

    @classmethod
    def rectangle_quad(cls, lo, hi, nx, ny):
        h = C.c_void_p()
        check(lib.femo_mesh_create_rectangle_quad(int(nx), int(ny), (C.c_double * 2)(*lo), (C.c_double * 2)(*hi), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = (nx, ny), tuple(lo), tuple(hi)
        return m

    @classmethod
    def from_arrays(cls, kind, coords, cells):
        """Unstructured mesh: kind 'interval' | 'triangle' | 'quadrilateral' | 'hexahedron', coords (nverts, gdim),
        cells (ncells, vertices per cell) in basix vertex order."""
        k = {'interval': 1, 'triangle': 2, 'quadrilateral': 3, 'hexahedron': 4}[kind]
        coords = np.ascontiguousarray(coords, dtype=np.float64)
        cells = np.ascontiguousarray(cells, dtype=np.int32)
        h = C.c_void_p()
        check(lib.femo_mesh_create_from_arrays(k, coords.shape[1], coords.shape[0], coords.ctypes.data_as(_DP_T), cells.shape[0],
                                               cells.ctypes.data_as(_I32P_T), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = None, tuple(coords.min(axis=0)), tuple(coords.max(axis=0))
        return m

    @classmethod
    def box_hex(cls, lo, hi, nx, ny, nz):
        h = C.c_void_p()
        check(lib.femo_mesh_create_box_hex(int(nx), int(ny), int(nz), (C.c_double * 3)(*lo), (C.c_double * 3)(*hi), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = (nx, ny, nz), tuple(lo), tuple(hi)
        return m

    @classmethod
    def interval(cls, n, x0, x1):
        h = C.c_void_p()
        check(lib.femo_mesh_create_interval(int(n), float(x0), float(x1), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = (n,), (x0,), (x1,)
        return m

    @classmethod
    def annulus(cls, nr, nth, r0=0.06, r1=0.12):
        h = C.c_void_p()
        check(lib.femo_mesh_create_annulus(int(nr), int(nth), float(r0), float(r1), C.byref(h)))
        m = cls(h)
        m.shape, m.lo, m.hi = (nr, nth), (r0, 0.0), (r1, 2 * np.pi)
        return m

    def coords(self):
        out = np.empty((self.nverts, self.gdim), dtype=np.float64)
        check(lib.femo_mesh_copy(self._h, 0, _np_ptr(out)))
        return out

    def cells(self):
        out = np.empty((self.ncells, self.nvpc), dtype=np.int32)
        check(lib.femo_mesh_copy(self._h, 1, _np_ptr(out)))
        return out

    def exterior_facets(self):
        c = np.empty(self.nbfacets, dtype=np.int32)
        l = np.empty(self.nbfacets, dtype=np.int32)
        check(lib.femo_mesh_copy(self._h, 2, _np_ptr(c)))
        check(lib.femo_mesh_copy(self._h, 3, _np_ptr(l)))
        return c, l

    def __del__(self):
        if getattr(self, '_h', None) and lib is not None:
            lib.femo_mesh_destroy(self._h)
            self._h = None


class EngineProblem:
    """One form family instantiated on a mesh: dofmaps, CSR patterns and gather
    maps on the host; after `upload()` the device-resident assembly / solve path."""

    def __init__(self, mesh, family, params=(), tagged=None, facets=None, cell_tags=None):
        self.mesh = mesh
        self.family = family
        h = C.c_void_p()
        pa = (C.c_double * max(1, len(params)))(*params)
        if facets is not None or cell_tags is not None:
            # general form: explicit one-sided facets (cell, local facet) and / or a subdomain id per cell
            fc = fl = tg = None
            nf = 0
            if facets is not None:
                fc = np.ascontiguousarray(facets[0], dtype=np.int32).ravel()
                fl = np.ascontiguousarray(facets[1], dtype=np.int32).ravel()
                nf = fc.size
            if cell_tags is not None:
                tg = np.ascontiguousarray(cell_tags, dtype=np.int32).ravel()
                assert tg.size == mesh.ncells
            check(lib.femo_problem_create_ex(mesh._h, int(family), pa, len(params),
                                             None if fc is None else _np_ptr(fc), None if fl is None else _np_ptr(fl),
                                             nf, None if tg is None else _np_ptr(tg), C.byref(h)))
        elif tagged is None:
            check(lib.femo_problem_create(mesh._h, int(family), pa, len(params), C.byref(h)))
        else:   # facets of a tagged measure ds(tag): indices into mesh.exterior_facets()
            tg = np.ascontiguousarray(tagged, dtype=np.int32).ravel()
            check(lib.femo_problem_create_tagged(mesh._h, int(family), pa, len(params), _np_ptr(tg), tg.size,
                                                 C.byref(h)))
        self._h = h
        s = (C.c_int64 * 16)()
        check(lib.femo_problem_sizes(self._h, s))
        self.N, self.nin, self.naux, self.nout = int(s[0]), int(s[1]), int(s[2]), int(s[3])
        self.M = [int(s[4 + i]) for i in range(self.nin)]
        self.aux_sizes = [int(s[8 + i]) for i in range(self.naux)]
        self.uploaded = False
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._keep = {}       # tensors whose pointers the engine borrows
        self._pinned = {}
        self.device = None

    # -- host-side layout queries ----------------------------------------
    def edges(self):
        """P2 states: (edge -> vertices (nedges,2), cell -> edges (ncells,3)) of the problem's mesh."""
        s = (C.c_int64 * 6)()
        check(lib.femo_problem_mesh_sizes(self._h, s))
        ncells, nverts = int(s[0]), int(s[1])
        ne = self.N - nverts
        ev = np.empty((ne, 2), dtype=np.int32)
        ce = np.empty((ncells, 3), dtype=np.int32)
        check(lib.femo_problem_mesh_copy(self._h, 4, ev.ctypes.data_as(C.c_void_p)))
        check(lib.femo_problem_mesh_copy(self._h, 5, ce.ctypes.data_as(C.c_void_p)))
        return ev, ce

    def pattern_info(self, which):
        info = (C.c_int64 * 4)()
        check(lib.femo_problem_pattern_info(self._h, which, info))
        return dict(rows=int(info[0]), cols=int(info[1]), nnz=int(info[2]), ncontrib=int(info[3]))

    def pattern(self, which):
        i = self.pattern_info(which)
        rowptr = np.empty(i['rows'] + 1, dtype=np.int32)
        col = np.empty(i['nnz'], dtype=np.int32)
        check(lib.femo_problem_pattern(self._h, which, _np_ptr(rowptr), _np_ptr(col)))
        return rowptr, col

    def gather_map(self, which):
        i = self.pattern_info(which)
        ptr = np.empty(i['nnz'] + 1, dtype=np.int32)
        src = np.empty(i['ncontrib'], dtype=np.int32)
        check(lib.femo_problem_gather_map(self._h, which, _np_ptr(ptr), _np_ptr(src)))
        return ptr, src

    def set_bc(self, dof_lists, g=None):
        dof_lists = [np.ascontiguousarray(d, dtype=np.int32).ravel() for d in dof_lists]
        ptr = np.zeros(len(dof_lists) + 1, dtype=np.int32)
        ptr[1:] = np.cumsum([d.size for d in dof_lists])
        dofs = np.concatenate(dof_lists) if dof_lists else np.zeros(0, dtype=np.int32)
        dofs = np.ascontiguousarray(dofs, dtype=np.int32)
        gp = None
        if g is not None:
            g = np.ascontiguousarray(np.broadcast_to(np.asarray(g, dtype=np.float64), (self.N,)))
            gp = _np_ptr(g)
        check(lib.femo_problem_set_bc(self._h, _np_ptr(dofs), _np_ptr(ptr), len(dof_lists), gp))

    def enable_multigrid(self):
        """Build the coarse-level layouts of the GMG preconditioner (host only, before upload)."""
        check(lib.femo_problem_enable_multigrid(self._h))
        self.mg_levels = lib.femo_problem_mg_levels(self._h)
        return self.mg_levels

    # -- device ------------------------------------------------------------
    def upload(self, device=0):
        import torch
        if not torch.cuda.is_available() or device_count() == 0:
            raise _lib.FemoError(-2, 'femo_b200 needs a CUDA device (sm_100a); there is no CPU path')
        self.device = torch.device('cuda', device)
        sb, wb = C.c_size_t(), C.c_size_t()
        check(lib.femo_problem_device_bytes(self._h, C.byref(sb), C.byref(wb)))
        self._static = torch.empty(sb.value, dtype=torch.uint8, device=self.device)
        self._work = torch.empty(wb.value, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
        check(lib.femo_problem_upload(self._h, device, C.c_void_p(stream), C.c_void_p(self._static.data_ptr()),
                                      sb.value, C.c_void_p(self._work.data_ptr()), wb.value))
        self.uploaded = True
        self.static_bytes, self.work_bytes = sb.value, wb.value
        return self

    def new_vector(self, n, fill=None):
        import torch
        if fill is None:
            return torch.empty(n, dtype=torch.float64, device=self.device)
        return torch.full((n,), float(fill), dtype=torch.float64, device=self.device)

    def pinned_buffer(self, n):
        """Pinned host staging buffer of n doubles (ring of three per size)."""
        import torch
        ring = self._pinned.setdefault(n, [[], 0])
        if len(ring[0]) < 3:
            ring[0].append(torch.empty(n, dtype=torch.float64).pin_memory().numpy())
            return ring[0][-1]
        ring[1] = (ring[1] + 1) % 3
        return ring[0][ring[1]]

    def to_device(self, array):
        import torch
        return torch.as_tensor(np.ascontiguousarray(array, dtype=np.float64)).to(self.device)

    def set_coefficient(self, slot, tensor):
        assert tensor.dtype.is_floating_point and tensor.element_size() == 8 and tensor.is_contiguous()
        check(lib.femo_set_coefficient(self._h, slot, C.c_void_p(tensor.data_ptr()), tensor.numel()))
        self._keep[slot] = tensor

    def coefficient(self, slot):
        return self._keep.get(slot)

    def set_param(self, index, value):
        check(lib.femo_problem_set_param(self._h, int(index), float(value)))

    def launch_count(self):
        n = C.c_longlong()
        check(lib.femo_problem_launch_count(self._h, C.byref(n)))
        return n.value

    def graph_replays(self):
        n = C.c_longlong()
        check(lib.femo_problem_graph_replays(self._h, C.byref(n)))
        return n.value

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def assemble_residual(self, out=None):
        out = self.new_vector(self.N) if out is None else out
        check(lib.femo_assemble_residual(self._h, self._p(out)))
        return out

    def assemble_jacobian(self, plain=True, bc=False, out=None, out_bc=None):
        nnz = self.pattern_info(0)['nnz']
        if plain and out is None:
            out = self.new_vector(nnz)
        if bc and out_bc is None:
            out_bc = self.new_vector(nnz)
        check(lib.femo_assemble_jacobian(self._h, self._p(out), self._p(out_bc)))
        return out, out_bc

    def assemble_dRdm(self, slot, out=None):
        out = self.new_vector(self.pattern_info(1 + slot)['nnz']) if out is None else out
        check(lib.femo_assemble_dRdm(self._h, slot, self._p(out)))
        return out

    def newton_rhs(self, vals, out=None):
        out = self.new_vector(self.N) if out is None else out
        check(lib.femo_newton_rhs(self._h, self._p(vals), self._p(out)))
        return out

    def system_rhs(self, vals, out=None):
        out = self.new_vector(self.N) if out is None else out
        check(lib.femo_assemble_system_rhs(self._h, self._p(vals), self._p(out)))
        return out

    def assemble_output(self, k=0):
        v = C.c_double()
        check(lib.femo_assemble_output(self._h, k, C.byref(v)))
        return v.value

    def assemble_output_grad(self, k, slot, out=None):
        n = self.N if slot == 0 else self.M[slot - 1]
        out = self.new_vector(n) if out is None else out
        check(lib.femo_assemble_output_grad(self._h, k, slot, self._p(out)))
        return out

    def assemble_output_and_grad(self, k=0, out=None):
        """J_k and dJ_k/du in one quadrature pass; returns (J, dJdu tensor)."""
        out = self.new_vector(self.N) if out is None else out
        v = C.c_double()
        check(lib.femo_assemble_output_and_grad(self._h, k, C.byref(v), self._p(out)))
        return v.value, out

    def spmv(self, which, vals, x, transpose=False, out=None):
        i = self.pattern_info(which)
        n = i['cols'] if transpose else i['rows']
        out = self.new_vector(n) if out is None else out
        check(lib.femo_spmv(self._h, which, self._p(vals), self._p(x), self._p(out), 1 if transpose else 0))
        return out

    def vcycle_op_probe(self, mode):
        """One launch of a fine-level V-cycle kernel (bench.py roofline); returns (algorithmic bytes, fine-level launches of
        this mode so far).  Modes: 0 residual, 1 / 2 Chebyshev steps, 3 fused pre-smoother (fp32 DIA planes), 4 / 5 fp64
        DIA SpMV with / without the fused dot, 6 / 7 down / up level sweep (smoother, residual and transfer fused)."""
        info = (C.c_int64 * 2)()
        check(lib.femo_vcycle_op_probe(self._h, int(mode), info))
        return int(info[0]), int(info[1])

    def spmv_bsr3(self, vals, x, out=None, convert=True):
        """y = A x through the 3x3-block copy of the dR/du values (3-component vertex states)."""
        out = self.new_vector(self.N) if out is None else out
        check(lib.femo_spmv_bsr3(self._h, self._p(vals), self._p(x), self._p(out), 1 if convert else 0))
        return out

    def axpy(self, a, x, y):
        check(lib.femo_axpy(self._h, float(a), self._p(x), self._p(y), x.numel()))
        return y

    # -- algebraic multigrid (precond 4): meshes without a lattice hierarchy ------------------------------------
    AMG_ARRAYS = ('rowptr', 'col', 'agg', 'p_rowptr', 'p_col', 'pp_ptr', 'pp_src', 'r_rowptr', 'r_col', 'r_perm',
                  'ap_rowptr', 'ap_col', 'ap_ptr', 'ap_ia', 'ap_ib', 'ac_ptr', 'ac_ia', 'ac_ib')
    AMG_VALUES = ('vals', 'p_vals', 'ap_vals', 'dinv')

    def amg_symbolic(self, vals=None, theta=-1.0, theta_decay=0.0, max_levels=0, coarse_size=0, block=0, omega_scale=None):
        """Pattern phase of the smoothed-aggregation hierarchy (host only).  vals: host copy of a BC'd Jacobian for
        the strength-of-connection test (None: every connection strong).  Returns levels / bytes / complexity."""
        from ._lib import AmgOpts
        o = AmgOpts(theta=theta, theta_decay=theta_decay, max_levels=max_levels, coarse_size=coarse_size, block=block,
                    omega_scale_set=0 if omega_scale is None else 1, omega_scale=0.0 if omega_scale is None else float(omega_scale))
        vp = None
        if vals is not None:
            vals = np.ascontiguousarray(vals, dtype=np.float64)
            assert vals.size == self.pattern_info(0)['nnz']
            vp = _np_ptr(vals)
        info = (C.c_int64 * 4)()
        check(lib.femo_amg_symbolic(self._h, vp, C.byref(o), info))
        self.amg = dict(levels=int(info[0]), bytes=int(info[1]), total_nnz=int(info[2]), coarsest=int(info[3]),
                        operator_complexity=int(info[2]) / float(self.pattern_info(0)['nnz']))
        return self.amg

    def amg_attach(self):
        """Upload the index lists of the hierarchy into a device buffer of this problem's device."""
        import torch
        self._amg_arena = torch.empty(self.amg['bytes'], dtype=torch.uint8, device=self.device)
        check(lib.femo_amg_attach(self._h, C.c_void_p(self._amg_arena.data_ptr()), self.amg['bytes']))
        return self

    def enable_amg(self, vals=None, **kw):
        """amg_symbolic + amg_attach; vals may be a device tensor (copied to the host for the strength test)."""
        if vals is not None and hasattr(vals, 'cpu'):
            vals = vals.cpu().numpy()
        self.amg_symbolic(vals, **kw)
        return self.amg_attach()

    def amg_numeric(self, vals):
        check(lib.femo_amg_numeric(self._h, self._p(vals)))

    def amg_level_info(self, level):
        info, dinfo = (C.c_int64 * 8)(), (C.c_double * 2)()
        check(lib.femo_amg_level_info(self._h, level, info, dinfo))
        keys = ('n', 'nnz', 'nc', 'nnzP', 'nnzAP', 'pairs_ap', 'pairs_ac', 'p_sources')
        d = {k: int(info[i]) for i, k in enumerate(keys)}
        d['lmax_host'], d['lmax_device'] = float(dinfo[0]), float(dinfo[1])
        return d

    def amg_level_array(self, level, name):
        i = self.amg_level_info(level)
        sizes = dict(rowptr=i['n'] + 1, col=i['nnz'], agg=i['n'] if i['nc'] else 0, p_rowptr=i['n'] + 1, p_col=i['nnzP'],
                     pp_ptr=i['nnzP'] + 1, pp_src=i['p_sources'], r_rowptr=i['nc'] + 1, r_col=i['nnzP'], r_perm=i['nnzP'],
                     ap_rowptr=i['n'] + 1, ap_col=i['nnzAP'], ap_ptr=i['nnzAP'] + 1, ap_ia=i['pairs_ap'], ap_ib=i['pairs_ap'],
                     ac_ia=i['pairs_ac'], ac_ib=i['pairs_ac'])
        if name == 'ac_ptr':
            n = self.amg_level_info(level + 1)['nnz'] + 1
        else:
            n = sizes[name] if (i['nc'] or name in ('rowptr', 'col')) else 0
        out = np.empty(n, dtype=np.int32)
        check(lib.femo_amg_level_array(self._h, level, self.AMG_ARRAYS.index(name), _np_ptr(out), n))
        return out

    def amg_level_values(self, level, name, from_device=False):
        i = self.amg_level_info(level)
        n = dict(vals=i['nnz'], p_vals=i['nnzP'], ap_vals=i['nnzAP'], dinv=i['n'])[name]
        out = np.empty(n, dtype=np.float64)
        check(lib.femo_amg_level_values(self._h, level, self.AMG_VALUES.index(name), 1 if from_device else 0, _np_ptr(out), n))
        return out

    def linear_solve(self, vals, b, x=None, transpose=False, rtol=1e-10, atol=0.0, max_it=100000, check_every=1,
                     precond=0, cheb_degree=0, cheb_ratio=0.0, method=0, restart=0, mg_precision=0):
        """method 0 = CG, 1 = restarted GMRES (non-symmetric Jacobians)."""
        x = self.new_vector(self.N, 0.0) if x is None else x
        o = KrylovOpts(rtol=rtol, atol=atol, max_it=max_it, precond=precond, cheb_degree=cheb_degree, method=method,
                       restart=restart, check_every=check_every, cheb_ratio=cheb_ratio, mg_precision=mg_precision)
        info = KrylovInfo()
        check(lib.femo_linear_solve(self._h, self._p(vals), self._p(b), self._p(x), 1 if transpose else 0,
                                    C.byref(o), C.byref(info)))
        return x, dict(iterations=info.iterations, converged=bool(info.converged), rnorm=info.rnorm,
                       bnorm=info.bnorm, spmv_count=info.spmv_count)

    def newton_solve(self, kind='Newton', atol=None, rtol=None, stol=1e-8, max_it=None, krylov_rtol=1e-10,
                     krylov_max_it=100000, check_every=1, precond=0, cheb_degree=0, cheb_ratio=0.0, method=0,
                     mg_precision=0, forcing=0.0):
        """kind 'Newton' = dolfinx NewtonSolver defaults of the reference (3 fixed
        iterations, utils_dolfinx.py:419-425); 'SNES' = PETSc newtonls (:376-416)."""
        snes = (kind == 'SNES')
        o = NewtonOpts()
        o.kind = 1 if snes else 0
        o.atol = (1e-13 if snes else 1e-50) if atol is None else atol
        o.rtol = (1e-13 if snes else 1e-30) if rtol is None else rtol
        o.stol = stol
        o.max_it = (100 if snes else 3) if max_it is None else max_it
        o.krylov = KrylovOpts(rtol=krylov_rtol, atol=0.0, max_it=krylov_max_it, precond=precond,
                              cheb_degree=cheb_degree, method=method, restart=0, check_every=check_every,
                              cheb_ratio=cheb_ratio, mg_precision=mg_precision, forcing=forcing)
        info = NewtonInfo()
        check(lib.femo_newton_solve(self._h, C.byref(o), C.byref(info)))
        return dict(iterations=info.iterations, converged=info.converged, fnorm0=info.fnorm0, fnorm=info.fnorm,
                    krylov_iterations=info.krylov_iterations, spmv_count=info.spmv_count)

    def __del__(self):
        if getattr(self, '_h', None) and lib is not None:
            lib.femo_problem_destroy(self._h)
            self._h = None
