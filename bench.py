#!/usr/bin/env python
"""bench.py -- state+adjoint solves/s on BASELINE.json's configs[1]:
nonlinear Poisson (examples/nonlinear_poisson_opt), P1 on the unit square,
n = 4000 (16 008 001 dofs, 32 000 000 cells, 112 024 001 nnz), f = 0.1, u0 = 0.

One step = what one optimiser gradient evaluation triggers (SURVEY.md section 8d):
SNES state solve (per Newton iteration: residual + Jacobian assembly + Krylov
solve), linearisation (dR/du, dR/dm), output J, dJ/du, dJ/dm, one transposed
(adjoint) Krylov solve and the dR/dm^T lambda product.

  value  engine-level step, every input resident in HBM, CUDA events
  e2e    the same step through the reference-facing API (FEAModel + Simulator:
         numpy in, numpy out), host<->device copies inside the timed region
  --impl reference   oracle/cpu_path.cpp, the C++/OpenMP restatement of the same step (the reference's
         dolfinx + MUMPS path is not installable offline) on all host cores, full workload size
  --workload p2|hex|motor   the P2 variant, the 3-D cantilever (configs[3]) and the chained motor problem
         (configs[4]) on one GPU (hex also on N), each verified by residual norms + a finite difference

Usage: python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--n 4000] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'state+adjoint solves/s'
UNIT = 'solves/s'
N_DEFAULT = 4000
N_DIST = 4096          # per-rank lattice of the multi-GPU runs (partitioned multigrid needs powers of two)
KRYLOV_RTOL = 1e-10


def workload(n, kind='p1'):
    if kind == 'p2':
        dofs = (n + 1) ** 2 + 2 * n * (n + 1) + n * n
        return dict(workload='nonlinear_poisson_opt P2 unit square n=%d (%d dofs, %d cells), SNES + adjoint, f=0.1, u0=0'
                    % (n, dofs, 2 * n * n), n=n, dofs=dofs, cells=2 * n * n,
                    solver='SNES newtonls atol=rtol=1e-13; p-multigrid (P2 -> P1 -> lattice hierarchy) preconditioned CG '
                           'rtol=%g replaces LU(MUMPS)' % KRYLOV_RTOL,
                    cache='working set exceeds the 126 MB L2; no explicit flush')
    if kind == 'motor':
        nr, nth = n, 4 * n
        dofs = (nr + 1) * nth
        return dict(workload='em_motor_opt on the synthetic annulus %dx%d (magnetostatics %d dofs + mesh motion %d dofs, %d cells, '
                             '216-subdomain tag layout): edge displacement -> mesh motion (2-step incremental SNES) -> '
                             'magnetostatics (5-step load ramp, SNES) -> B influence, chained EM + mesh-motion adjoints'
                             % (nr, nth, dofs, 2 * dofs, 2 * nr * nth), n=n, dofs=3 * dofs, cells=2 * nr * nth,
                    solver='SNES newtonls, inexact (Eisenstat-Walker forcing, eta_max --forcing); GMRES(70) right-preconditioned by a '
                           'smoothed-aggregation AMG V-cycle, adjoints to rtol=%g; replaces LU(MUMPS)' % KRYLOV_RTOL,
                    cache='working set exceeds the 126 MB L2; no explicit flush')
    if kind == 'hex':
        nx, ny, nz = n, n // 2, n // 4
        dofs = 3 * (nx + 1) * (ny + 1) * (nz + 1)
        return dict(workload='beam_topo_opt 3-D hexahedral SIMP cantilever %dx%dx%d (%d dofs, %d cells), Newton (3 fixed '
                             'iterations, reference-faithful) + compliance adjoint, density = cone filter (beta 2) of 0.86*random(nel), '
                             'np.random.seed(0), bounds [1e-4,1]' % (nx, ny, nz, dofs, nx * ny * nz), n=n, dofs=dofs, cells=nx * ny * nz,
                    solver='NewtonSolver max_it=3; GMG-preconditioned CG rtol=%g replaces LU(MUMPS)' % KRYLOV_RTOL,
                    cache='working set exceeds the 126 MB L2; no explicit flush')
    return dict(workload='nonlinear_poisson_opt P1 unit square n=%d (%d dofs, %d cells), SNES + adjoint, f=0.1, u0=0'
                % (n, (n + 1) ** 2, 2 * n * n), n=n, dofs=(n + 1) ** 2, cells=2 * n * n,
                solver='SNES newtonls atol=rtol=1e-13; GMG-preconditioned CG rtol=%g replaces LU(MUMPS)' % KRYLOV_RTOL,
                cache='working set (>10 GB) exceeds the 126 MB L2; no explicit flush')


def base_dofs_of(n, kind):
    return (n + 1) ** 2 if kind in ('p1', 'motor') else 3 * (n + 1) * (n // 2 + 1) * (n // 4 + 1)


def global_dofs_of(n, kind, world):
    """dofs of the ONE partitioned problem `--gpus world` runs (EngineStep builds exactly this)."""
    if world == 1:
        return workload(n, kind)['dofs']
    if kind == 'hex':
        return 3 * (n + 1) * (n // 2 + 1) * (n // 4 * world + 1)
    return (N_DIST + 1) * (N_DIST * world + 1)


def arm_config(n, kind, world):
    """`config` of the JSON line, one function for BOTH arms: `--impl reference` must describe the same workload as the
    femo_b200 arm launched with the same flags."""
    cfg = workload(n, kind)
    gd = global_dofs_of(n, kind, world)
    if world > 1:
        cfg['workload'] = ('weak-scaled %s: %d dofs over %d GPUs (the N=1 workload has %d)'
                           % (cfg['workload'].split(' n=')[0] if kind == 'p1' else cfg['workload'].split(' (')[0],
                              gd, world, base_dofs_of(n, kind)))
        cfg['dofs'] = gd
    cfg['parallelism'] = ('1 GPU' if world == 1 else
                          (('one cantilever of %d x %d x %d cells (%d dofs), z-slab partition ' % (n, n // 2, n // 4 * world, gd))
                           if kind == 'hex' else
                           ('one problem on [0,1]x[0,%d], %d x %d cells (%d dofs), y-slab partition ' % (world, N_DIST, N_DIST * world, gd))) +
                          ('with one-cell ghost layer over %d GPUs, halo exchange + all-reduce, '
                           'partitioned multigrid; value = solves/s x dofs/dofs(N=1 workload)' % world))
    return cfg


# ---------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------
# engine-level step (inputs resident in HBM)
# ---------------------------------------------------------------------------
class EngineStep:
    """world == 1: the n x n unit-square problem on one GPU.
    world > 1: ONE problem on [0,1] x [0,world] with N_DIST x (N_DIST*world) cells (weak scaling, square
    cells), cut into y-slabs: rank r owns N_DIST cell rows + a one-cell ghost layer; halo exchange per
    SpMV, all-reduced Krylov/Newton scalars, partitioned multigrid -- all inside libfemo_b200 over NCCL."""

    def __init__(self, n, device, rank=0, world=1, kind='p1'):
        import torch
        from femo_b200 import engine as E
        self.torch = torch
        self.kind = kind
        self.out_id = 0
        if kind == 'hex' and world > 1:
            # weak scaling of ONE cantilever: nx x ny x (nz*world) cells cut into z-slabs (SURVEY.md section 8e)
            import numpy as np
            from femo_b200 import dist as fd
            nx, ny, nz = n, n // 2, n // 4
            gnz = nz * world
            p = fd.SlabProblem(E.FAMILY_SIMP_HEX8, nx, gnz, rank, world, lo=(0.0, 0.0, 0.0), hi=(2.0 * nx, 2.0 * ny, 2.0 * gnz),
                               params=[0.3, 0.0, -0.25, 0.0, 3.0], ny=ny, face_mask=1 << 3)
            xl = p.local_coords()
            nodes = np.nonzero(xl[:, 0] == 0.0)[0]
            p.set_bc([np.stack([3 * nodes, 3 * nodes + 1, 3 * nodes + 2], axis=1).ravel().astype(np.int32)])
            self.global_dofs = 3 * (nx + 1) * (ny + 1) * (gnz + 1)
            self.out_id = 1
        elif kind == 'hex':
            import numpy as np
            nx, ny, nz = n, n // 2, n // 4
            mesh = E.EngineMesh.box_hex((0.0, 0.0, 0.0), (2.0 * nx, 2.0 * ny, 2.0 * nz), nx, ny, nz)
            fc, fl = mesh.exterior_facets()
            p = E.EngineProblem(mesh, E.FAMILY_SIMP_HEX8, [0.3, 0.0, -0.25, 0.0, 3.0],
                                tagged=np.nonzero(fl == 3)[0].astype(np.int32))         # traction on x = Lx
            nodes = np.arange((ny + 1) * (nz + 1)) * (nx + 1)                           # clamp x = 0
            p.set_bc([np.stack([3 * nodes, 3 * nodes + 1, 3 * nodes + 2], axis=1).ravel().astype(np.int32)])
            self.global_dofs = 3 * (nx + 1) * (ny + 1) * (nz + 1)
            self.out_id = 1                                                              # compliance
        elif kind == 'p2':
            p = E.EngineProblem(E.EngineMesh.unit_square(n), E.FAMILY_NLPOISSON_P2)
            self.global_dofs = (n + 1) ** 2 + 2 * n * (n + 1) + n * n
        elif world == 1:
            p = E.EngineProblem(E.EngineMesh.unit_square(n), E.FAMILY_NLPOISSON_P1)
            self.global_dofs = (n + 1) ** 2
        else:
            from femo_b200 import dist as fd
            p = fd.SlabProblem(E.FAMILY_NLPOISSON_P1, N_DIST, N_DIST * world, rank, world, lo=(0.0, 0.0),
                               hi=(1.0, float(world)))
            self.global_dofs = (N_DIST + 1) * (N_DIST * world + 1)
        p.enable_multigrid()
        p.upload(device)
        self.p = p
        self.u = p.new_vector(p.N, 0.0)
        if kind == 'hex':
            import numpy as np
            nx, ny, nz = n, n // 2, n // 4
            # the reference's initial design (run_topo_opt_cantilever_beam.py:175-180): np.random.seed(0),
            # density_unfiltered = 0.86 * random(nel) within the design bounds [1e-4, 1], passed through the cone filter
            # of the pre-processor (general_filter_model.py:67-90, beta = 2, h_avg = cell size) before it enters the PDE
            import ctypes as C
            from femo_b200._lib import lib, check
            gnz = nz * world
            np.random.seed(0)
            unf = np.clip(0.86 * np.random.random(nx * ny * gnz), 1e-4, 1.0)
            d_unf, d_rho, d_den = p.to_device(unf), p.new_vector(unf.size), p.new_vector(unf.size)
            check(lib.femo_filter_apply3(device, C.c_void_p(torch.cuda.current_stream().cuda_stream), nx, ny, gnz, 2.0, 2.0, 2.0,
                                         4.0, C.c_void_p(d_unf.data_ptr()), C.c_void_p(d_rho.data_ptr()),
                                         C.c_void_p(d_den.data_ptr()), 0))
            if world > 1:
                s = p.slab
                d_rho = d_rho.reshape(gnz, nx * ny)[s['crow0']:s['crow0'] + s['ncrows']].reshape(-1)
            self.f = d_rho.contiguous().clone()
            del d_unf, d_den
        else:
            self.f = p.new_vector(p.M[0], 0.1)
        p.set_coefficient(0, self.u)
        p.set_coefficient(1, self.f)
        nnz = p.pattern_info(0)['nnz']
        self.nnz = nnz
        self.vals = p.new_vector(nnz)
        self.vals_bc = p.new_vector(nnz) if kind == 'hex' else None
        self.dv = p.new_vector(p.pattern_info(1)['nnz'])
        self.dJdu = p.new_vector(p.N)
        self.grad = p.new_vector(p.M[0])
        self.lam = p.new_vector(p.N)
        self.tmp = p.new_vector(p.M[0])
        self.info = {}

    def launch_count(self):
        return self.p.launch_count()

    def step(self):
        p = self.p
        k = self.out_id
        self.u.zero_()                                        # same work every step (cudaMemset, not a kernel of ours)
        if self.kind == 'hex':     # linear problem through the reference's NewtonSolver (3 fixed iterations, quirk B1)
            ni = p.newton_solve(kind='Newton', krylov_rtol=KRYLOV_RTOL, precond=2, cheb_degree=2)
            p.assemble_jacobian(plain=True, bc=True, out=self.vals, out_bc=self.vals_bc)
        else:
            ni = p.newton_solve(kind='SNES', krylov_rtol=KRYLOV_RTOL, precond=2, cheb_degree=2)
            p.assemble_jacobian(plain=True, bc=False, out=self.vals)      # dR/du at the converged state
        p.assemble_dRdm(0, self.dv)                                        # dR/df
        J, _ = p.assemble_output_and_grad(k, self.dJdu)                   # objective (host scalar) + dJ/du, one pass
        p.assemble_output_grad(k, 1, self.grad)
        self.lam.zero_()
        _, li = p.linear_solve(self.vals_bc if self.kind == 'hex' else self.vals, self.dJdu, self.lam, transpose=True,
                               rtol=KRYLOV_RTOL, precond=2, cheb_degree=2)
        p.spmv(1, self.dv, self.lam, transpose=True, out=self.tmp)
        p.axpy(-1.0, self.tmp, self.grad)                                  # dJ/df = pJ/pf - dRdf^T lambda
        self.info = dict(newton_its=ni['iterations'], krylov_its=ni['krylov_iterations'], adjoint_its=li['iterations'],
                         fnorm0=ni['fnorm0'], fnorm=ni['fnorm'],
                         converged=(bool(ni['converged']) or self.kind == 'hex') and li['converged'], J=J)
        return J

    def outputs(self):
        """What the last step() returned to its caller: the objective, the state and dJ/df."""
        return dict(J=self.info['J'], u=self.u, dJdf=self.grad)


class MotorStep:
    """BASELINE.json configs[4] (examples/em_motor_opt/run_motor_opt.py:94-317) at engine level on the synthetic annulus:
    one step = mesh-motion state (2 incremental SNES solves) + magnetostatic state (5-step ramp of the sources) + the
    chained total derivative of the B-influence functional w.r.t. the prescribed edge displacement (EM adjoint solve,
    dR_em/duhat^T, mesh-motion adjoint solve, dR_mm/dg^T)."""
    kind = 'motor'

    def __init__(self, nr, device, precond='amg', forcing=0.0):
        import numpy as np
        import torch
        from femo_b200 import engine as E
        from femo_b200.forms import motor as pde
        from femo_b200.fea.fem import Mesh
        self.torch = torch
        nth = 4 * nr
        em = E.EngineMesh.annulus(nr, nth)
        mesh = Mesh(em, 'triangle')
        tags = pde.synthetic_motor_tags(mesh)
        mid = nr // 2
        sides = [pde.annulus_circle_sides(mesh, k) for k in (0, mid, nr)]
        fc, fl = np.concatenate([q[0] for q in sides]), np.concatenate([q[1] for q in sides])
        o = np.lexsort((fl, fc))
        self.mm = E.EngineProblem(em, E.FAMILY_MOTOR_MM, [5e3], facets=(fc[o], fl[o]), cell_tags=tags)
        self.em = E.EngineProblem(em, E.FAMILY_MOTOR_EM,
                                  pde.em_params(838.e3, 12, 36, 4e-7 * np.pi, 0.0, 282.2 / 0.00016231), cell_tags=tags)
        self.mm.upload(device)
        self.em.upload(device)
        self.p = self.em
        X = em.coords()
        g = np.zeros(2 * X.shape[0])
        nodes = mid * nth + np.arange(nth)
        frac = 0.1 * (0.06 / nr) / 0.09                      # the interior circle (r = 0.09) grows by a tenth of a radial cell
        g[2 * nodes], g[2 * nodes + 1] = frac * X[nodes, 0], frac * X[nodes, 1]
        self.g = self.mm.to_device(g)
        self.gs = self.mm.new_vector(g.size, 0.0)
        self.uhat = self.mm.new_vector(self.mm.N, 0.0)
        self.A = self.em.new_vector(self.em.N, 0.0)
        self.mm.set_coefficient(0, self.uhat); self.mm.set_coefficient(1, self.gs)
        self.em.set_coefficient(0, self.A); self.em.set_coefficient(1, self.uhat)
        self.global_dofs = self.mm.N + self.em.N
        self.nnz = self.em.pattern_info(0)['nnz']
        self.vals = self.em.new_vector(self.nnz)
        self.vals_mm = self.mm.new_vector(self.mm.pattern_info(0)['nnz'])
        self.vals_bc = None
        if precond == 'amg':
            self.kw = dict(method=1, precond=4, cheb_degree=2, cheb_ratio=4.0)
            t0 = time.perf_counter()
            self.em.set_param(6, 0.2)
            self.em.assemble_jacobian(out=self.vals)
            self.em.enable_amg(self.vals)
            self.mm.assemble_jacobian(out=self.vals_mm)
            self.mm.enable_amg(self.vals_mm, omega_scale=0.0)        # plain aggregation + degree-4 smoother (family.py)
            self.kw_mm = dict(method=1, precond=4, cheb_degree=4, cheb_ratio=8.0)
            self.setup = dict(seconds=time.perf_counter() - t0, em=self.em.amg, mm=self.mm.amg)
        else:
            self.kw = self.kw_mm = dict(method=1, precond=1, cheb_degree=24, cheb_ratio=600.0)
            self.setup = None
        self.forcing = float(forcing)
        self.info = {}

    def launch_count(self):
        return self.em.launch_count() + self.mm.launch_count()

    def step(self):
        em, mm, kw = self.em, self.mm, self.kw
        its = dict(mm_newton=0, mm_krylov=0, em_newton=0, em_krylov=0)
        self.uhat.zero_()
        for i in (1, 2):                                            # solveIncremental, run_motor_opt.py:120-142
            self.torch.mul(self.g, i / 2.0, out=self.gs)
            ni = mm.newton_solve(kind='SNES', krylov_rtol=KRYLOV_RTOL, krylov_max_it=40000, forcing=self.forcing, **self.kw_mm)
            its['mm_newton'] += ni['iterations']; its['mm_krylov'] += ni['krylov_iterations']
        self.A.zero_()
        for st in range(1, 6):                                      # solveIncrementalEM, :231-250
            em.set_param(6, st / 5.0)
            ne = em.newton_solve(kind='SNES', krylov_rtol=KRYLOV_RTOL, krylov_max_it=40000, forcing=self.forcing, **kw)
            its['em_newton'] += ne['iterations']; its['em_krylov'] += ne['krylov_iterations']
        em.assemble_jacobian(out=self.vals)
        J, dJdA = em.assemble_output_and_grad(0)
        lam_e, le = em.linear_solve(self.vals, dJdA, transpose=True, rtol=KRYLOV_RTOL, max_it=40000, **kw)
        dJduh = em.assemble_output_grad(0, 1)
        em.axpy(-1.0, em.spmv(1, em.assemble_dRdm(0), lam_e, transpose=True), dJduh)
        mm.assemble_jacobian(out=self.vals_mm)
        lam_m, lm = mm.linear_solve(self.vals_mm, dJduh, transpose=True, rtol=KRYLOV_RTOL, max_it=40000, **self.kw_mm)
        self.grad = mm.spmv(1, mm.assemble_dRdm(0), lam_m, transpose=True)
        self.grad.neg_()
        self.info = dict(its, krylov_its=its['em_krylov'] + its['mm_krylov'], adjoint_its=le['iterations'] + lm['iterations'],
                         em_adjoint_its=le['iterations'], mm_adjoint_its=lm['iterations'], newton_its=its['em_newton'] + its['mm_newton'],
                         converged=bool(ne['converged'] and ni['converged'] and le['converged'] and lm['converged']),
                         fnorm=ne['fnorm'], J=J)
        return J

    def outputs(self):
        """What the last step() returned to its caller: B-influence, both states and dJ/dg."""
        return dict(J=self.info['J'], A=self.A, uhat=self.uhat, dJdg=self.grad)


DUMP_SAMPLE = 1 << 20          # entries kept of a larger output over all ranks: at most 4 outputs x 8 MB = 32 MB a run


def dump_outputs(d, outputs, rank=0, world=1):
    """--dump-outputs: writes each output of the last timed step as d/<name>.npy (rank r of a multi-GPU run: <name>.rank<r>.npy)
    in float64.  An output of more than DUMP_SAMPLE // world entries is reduced to that many at sorted indices drawn from a
    fixed seed, the same indices every run, so that the files of two builds compare entry for entry."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    keep = DUMP_SAMPLE // world
    suffix = '' if world == 1 else '.rank%d' % rank
    for name, a in outputs.items():
        if hasattr(a, 'cpu'):                                    # device tensor: sample on the device, copy the sample
            import torch
            a = a.reshape(-1)
            if a.numel() > keep:
                a = a[torch.from_numpy(_sample(a.numel(), keep)).to(a.device)]
            a = a.cpu().numpy()
        else:
            a = np.ravel(a)
            if a.size > keep:
                a = a[_sample(a.size, keep)]
        np.save(os.path.join(d, name + suffix + '.npy'), np.asarray(a, dtype=np.float64))


def _sample(n, k):
    import numpy as np
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def verify(es):
    """Correctness of the timed configuration at its full size, outside the timed region: fp64 residual norm of the
    returned state, fp64 residual of the adjoint system, and a central finite difference of the reduced functional along
    a smooth direction against the adjoint gradient (BASELINE.json: derivatives cross-checked by finite differences)."""
    torch, p = es.torch, es.p
    if es.kind == 'motor':
        return verify_motor(es)
    es.step()
    g = es.grad.clone()
    R = p.assemble_residual()
    vals = es.vals_bc if es.vals_bc is not None else es.vals
    if es.vals_bc is not None:                       # Dirichlet rows of the residual are replaced by u - g in the solve
        R = p.newton_rhs(vals)
    fnorm = float(R.norm())
    res = p.spmv(0, vals, es.lam, transpose=True)
    res -= es.dJdu
    adj = float(res.norm()) / float(es.dJdu.norm())
    M = p.M[0]
    d = 1.0 + 0.5 * torch.sin(2 * torch.pi * torch.arange(M, device=g.device, dtype=torch.float64) / M)
    f0 = es.f.clone()
    h = 1e-4
    if es.kind == 'hex':                             # densities in [1e-4, 1]: a relative perturbation keeps them positive
        d = d * f0
        h = 1e-3
    gd = float(g @ d)
    es.f.copy_(f0 + h * d)
    Jp = es.step()
    es.f.copy_(f0 - h * d)
    Jm = es.step()
    es.f.copy_(f0)
    fd = (Jp - Jm) / (2 * h)
    out = dict(state_residual_norm=fnorm, adjoint_relative_residual=adj, dJdf_dot_d=gd, finite_difference=fd,
               fd_relative_error=abs(fd - gd) / abs(fd))
    out['ok'] = bool(fnorm <= 1e-6 * max(es.info['fnorm0'], 1e-300) and adj < 10 * KRYLOV_RTOL and out['fd_relative_error'] < 1e-5)
    return out


def verify_motor(es):
    """Chained motor step: residual norms of both states and a central finite difference of B-influence along a smooth
    scaling of the prescribed edge displacement against the chained adjoint gradient."""
    torch = es.torch
    es.step()
    g = es.grad.clone()
    r_mm, r_em = float(es.mm.assemble_residual().norm()), float(es.em.assemble_residual().norm())
    n = es.g.numel()
    d = es.g * (1.0 + 0.5 * torch.sin(2 * torch.pi * torch.arange(n, device=g.device, dtype=torch.float64) / n))
    gd = float(g @ d)
    g0 = es.g.clone()
    h = 1e-3
    es.g.copy_(g0 + h * d)
    Jp = es.step()
    es.g.copy_(g0 - h * d)
    Jm = es.step()
    es.g.copy_(g0)
    fd = (Jp - Jm) / (2 * h)
    out = dict(mesh_motion_residual_norm=r_mm, magnetostatic_residual_norm=r_em, dJdg_dot_d=gd, finite_difference=fd,
               fd_relative_error=abs(fd - gd) / max(abs(fd), 1e-300))
    out['ok'] = bool(out['fd_relative_error'] < 1e-4)
    return out


VCYCLE_KERNELS = {0: 'femo::k_dia_apply<DIA_PLAIN,7> (V-cycle residual r = b - A x, fp32 DIA planes)',
                  1: 'femo::k_dia_apply<DIA_CHEB0,7> (post-smoother first Chebyshev step)',
                  2: 'femo::k_dia_apply<DIA_CHEBK,7> (post-smoother second Chebyshev step)',
                  3: 'femo::k_dia_apply<DIA_PRE2,7> (fused zero-guess degree-2 pre-smoother)',
                  4: 'femo::k_dia_spmv64<DOT,7> (CG recurrence q = A p with fused p.q, fp64 DIA planes)',
                  5: 'femo::k_dia_spmv64<PLAIN,7> (fp64 residuals of the CG start and the full-multigrid levels)'}
PROBE_MODES = tuple(sorted(VCYCLE_KERNELS))


def _time_launches(torch, fn, reps):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def time_kernels(es, counts, steps, reps=50):
    """Average launch duration (CUDA events on the launching stream, inputs > L2) of the hot kernels at the fine
    level: the four instantiations of the V-cycle operator (fp32 DIA planes), the two of the fp64 DIA SpMV the CG
    recurrence applies, and the CSR-stream SpMV behind `femo_spmv` (the operator kernel of non-lattice problems).
    counts[mode] = fine-level launches during the timed steps (counted by the engine) -> share of the step."""
    torch, p = es.torch, es.p
    out = []
    if counts is not None:
        for mode in PROBE_MODES:
            alg, _ = p.vcycle_op_probe(mode)
            t = _time_launches(torch, lambda: p.vcycle_op_probe(mode), reps)
            out.append(dict(kernel=VCYCLE_KERNELS[mode], launch_ms=t * 1e3, algorithmic_bytes=alg,
                            launches_per_step=counts[mode] / float(steps)))
    x = p.new_vector(p.N, 1.0)
    y = p.new_vector(p.N)
    if es.kind == 'hex':      # the CG recurrence of 3-component states streams the 3x3-block copy of the values
        vv = es.vals_bc if es.vals_bc is not None else es.vals
        p.spmv_bsr3(vv, x, out=y, convert=True)
        t = _time_launches(torch, lambda: p.spmv_bsr3(vv, x, out=y, convert=False), reps)
        out.append(dict(kernel='femo::k_spmv_bsr3 (BSR-3 SpMV of the CG recurrence, fine-level Jacobian)', launch_ms=t * 1e3,
                        algorithmic_bytes=8 * es.nnz + 4 * (es.nnz // 9) + 16 * p.N + 4 * (p.N // 3),
                        launches_per_step=es.info.get('adjoint_its', 0) + 1.0))
    if es.kind == 'p1':
        # assembly of the fine-level Jacobian and residual (BASELINE.json: "assembly GB/s vs HBM").  Node-centric lattice
        # kernels: no scratch, no gather map, constant geometry -- algorithmic bytes = values written + u and f read once;
        # they are fp64-pipe bound (closed-form element rows, 6 cells per node), the HBM fraction is reported for scale
        nc = p.M[0]
        t = _time_launches(torch, lambda: p.assemble_jacobian(plain=True, bc=False, out=es.vals), max(5, reps // 5))
        out.append(dict(kernel='femo::k_nlpoisson_p1_node_jac (fine-level Jacobian assembly, CSR values; fp64-pipe bound)',
                        launch_ms=t * 1e3, algorithmic_bytes=8 * es.nnz + 8 * p.N + 8 * nc,
                        launches_per_step=es.info.get('newton_its', 0) + 1.0))
        t = _time_launches(torch, lambda: p.assemble_residual(y), max(5, reps // 5))
        out.append(dict(kernel='femo::k_nlpoisson_p1_node_res (fine-level residual assembly; fp64-pipe bound)',
                        launch_ms=t * 1e3, algorithmic_bytes=16 * p.N + 8 * nc,
                        launches_per_step=es.info.get('newton_its', 0) + 1.0))
    t = _time_launches(torch, lambda: p.spmv(0, es.vals, x, out=y), reps)
    # lattice P1 problems apply the fine-level operator from DIA planes (rows above): the CSR kernel is then not part of
    # the step; the other workloads run one per Krylov iteration plus the residual checks
    per_step = 0.0 if counts is not None else es.info.get('krylov_its', 0) + es.info.get('adjoint_its', 0) + 5.0
    out.append(dict(kernel='femo::k_spmv<double> (CSR-stream SpMV, fine-level Jacobian; femo_spmv and non-lattice operators)',
                    launch_ms=t * 1e3, algorithmic_bytes=12 * es.nnz + 20 * p.N, launches_per_step=per_step))
    return out


# ---------------------------------------------------------------------------
# API-level step (host buffers): the call a femo user makes
# ---------------------------------------------------------------------------
class ApiStep:
    def __init__(self, n, degree=1, pinned=True):
        import numpy as np
        from femo_b200.fea.fea_b200 import FEA, createUnitSquareMesh, FunctionSpace, Function, TestFunction
        from femo_b200.forms.nonlinear_poisson import pdeRes, outputForm
        from femo_b200.csdl_opt import FEAModel, Simulator
        from femo_b200.fea import utils_b200
        utils_b200.KRYLOV['rtol'] = KRYLOV_RTOL
        mesh = createUnitSquareMesh(n)
        fea = FEA(mesh)
        f = Function(FunctionSpace(mesh, ('DG', 0)))
        Vu = FunctionSpace(mesh, ('CG', degree))
        u = Function(Vu)
        res = pdeRes(u, TestFunction(Vu), f)
        fea.add_input('f', f)
        fea.add_state(name='u', function=u, residual_form=res, arguments=['f'])
        fea.add_output(name='l2_functional', type='scalar', form=outputForm(u, f), arguments=['f', 'u'])
        fea.PDE_SOLVER = 'SNES'
        fea.REPORT = False
        model = FEAModel(fea=[fea], debug_mode=False)
        model.create_input('f', shape=fea.inputs_dict['f']['shape'], val=0.1)
        self.sim = Simulator(model, pinned=pinned)
        self.f0 = np.full(fea.inputs_dict['f']['shape'], 0.1)
        self.u0 = np.zeros(fea.states_dict['u']['shape'])
        self.fam = res.fam
        self.np = np

    def step(self):
        sim = self.sim
        sim['f'] = self.f0                       # host input of this step
        sim['u'] = self.u0                       # same initial guess every step
        sim.run()
        g = sim.compute_totals('l2_functional', 'f')[('l2_functional', 'f')]
        return float(sim['l2_functional'][0]), g


# ---------------------------------------------------------------------------
# CPU arm: oracle/cpu_path.cpp, the C++/OpenMP restatement of the same step with the same GMG-PCG algorithm
# (the reference's dolfinx + MUMPS path is not installable offline), on all host cores, at the FULL workload size
# ---------------------------------------------------------------------------
def host_threads():
    """All host threads this process may use.  Passed explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers when
    it starts more than one, which would silently turn the CPU arm of a --gpus N run into a single-threaded one."""
    try:
        return max(len(os.sched_getaffinity(0)), 1)
    except AttributeError:
        return max(os.cpu_count() or 1, 1)


def cpu_step(n):
    from oracle import cpu_path
    t = time.perf_counter()
    r = cpu_path.step(n, 0.1, krylov_rtol=KRYLOV_RTOL, nthreads=host_threads())
    dt = time.perf_counter() - t
    if not r['converged']:
        raise RuntimeError('cpu_path: SNES / Krylov did not converge')
    return dt, r


def cpu_baseline(n, steps=1):
    """One warm-up (page faults of the persistent workspace) + `steps` timed state+adjoint solves at the full size."""
    cpu_step(n)
    ts = []
    for _ in range(steps):
        dt, r = cpu_step(n)
        ts.append(dt)
    t = sum(ts) / len(ts)
    return dict(value=1.0 / t, unit=UNIT, cores=r['threads'], kind='port',
                sample='oracle/cpu_path.cpp (C++/OpenMP, %d threads): %d full state+adjoint solve(s) at n=%d (%d dofs) after one '
                       'warm-up, %.2f s each, same SNES + FMG/GMG-PCG algorithm and tolerances as the GPU arm (Newton its %d, '
                       'Krylov its %d + %d), no extrapolation' % (r['threads'], steps, n, (n + 1) ** 2, t, r['newton_its'],
                                                                   r['krylov_its'], r['adjoint_its']),
                J=r['J'])


# ---------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='femo_b200')
    ap.add_argument('--n', type=int, default=N_DEFAULT)
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--workload', default='p1', choices=['p1', 'p2', 'hex', 'motor'],
                    help="p1 = BASELINE.json configs[1] (the metric's config, default); p2 / hex / motor = the P2 variant of "
                         "configs[1], the 3-D cantilever of configs[3] and the chained motor problem of configs[4], for profiles/")
    ap.add_argument('--precond', default='amg', choices=['amg', 'cheb'], help='motor workload: AMG V-cycle or the round-1 polynomial')
    ap.add_argument('--forcing', type=float, default=0.01, help='motor workload: eta_max of the Eisenstat-Walker inexact Newton (0: every linear solve to rtol)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned as DIR/<name>.npy (float64; an output of more '
                         'than %d entries / number of ranks as the same seeded sample every run, 32 MB at most in all; rank r of a '
                         'multi-GPU run writes <name>.rank<r>.npy)' % DUMP_SAMPLE)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.workload != 'p1':
        if a.n == N_DEFAULT:
            a.n = dict(p2=2000, hex=256, motor=512)[a.workload]
        a.no_cpu = True
        if a.workload in ('hex', 'motor'):
            a.no_e2e = True
        if a.workload == 'motor' and int(os.environ.get('WORLD_SIZE', '1')) > 1:
            raise SystemExit('the motor workload runs on one GPU')
        if a.workload == 'p2' and int(os.environ.get('WORLD_SIZE', '1')) > 1:
            raise SystemExit('the P2 workload runs on one GPU')
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    W = max(a.warmup, 3)

    if a.impl == 'reference':
        if rank != 0:
            return 0
        # every step is one FULL state+adjoint solve of the N=1 workload (n=4000, 16M dofs) on all host cores, about 3 - 4 s
        # each on the GPU box: --steps 20 --warmup 5 ends within two minutes.  Under --gpus N > 1 the femo_b200 arm solves ONE
        # N-times larger problem and normalises its value to solves of the N=1 workload; the bounded CPU sample of that
        # workload is the N=1-sized problem itself, in the same normalised unit, so `config` is the GPU arm's for the same flags
        wr = max(int(a.warmup), 1)
        for _ in range(wr):
            cpu_step(a.n)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            _, r = cpu_step(a.n)
        dt = (time.perf_counter() - t0) / a.steps
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, dict(J=r['J'], u=r['u'], dJdf=r['grad']))
        val = 1.0 / dt
        sample = ('oracle/cpu_path.cpp: C++/OpenMP restatement of the reference path (the reference itself needs dolfinx + '
                  'PETSc/MUMPS, not installable offline) with the GPU arm\'s algorithm (SNES + FMG/GMG-PCG rtol %g) on %d host '
                  'threads; every step is a full n=%d solve (%d dofs = the N=1 workload%s), %.2f s per state+adjoint solve, %d '
                  'warm-up(s), no extrapolation; J=%.13g, Newton its %d, Krylov its %d + %d'
                  % (KRYLOV_RTOL, r['threads'], a.n, (a.n + 1) ** 2,
                     '' if world == 1 else '; the %d-GPU arm\'s value is normalised to solves of this workload' % world,
                     dt, wr, r['J'], r['newton_its'], r['krylov_its'], r['adjoint_its']))
        print(json.dumps(dict(metric=METRIC, value=val, unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=wr,
                              ms_per_step=1e3 / val, higher_is_better=True, scaling='weak', vs_baseline=None,
                              dtype='f64', data='synthetic', config=arm_config(a.n, a.workload, max(world, a.gpus)),
                              impl='reference',
                              cpu_baseline=dict(value=val, unit=UNIT, cores=r['threads'], kind='port', sample=sample),
                              e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps(dict(metric=METRIC, error='no CUDA device; femo_b200 has no CPU path')))
        return 1
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world > 1:
        from femo_b200 import dist as fd
        fd.init(local_rank)
    es = MotorStep(a.n, local_rank, a.precond, a.forcing) if a.workload == 'motor' else EngineStep(a.n, local_rank, rank, world, a.workload)
    for _ in range(W):
        es.step()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    l0 = es.launch_count()
    has_dia = a.workload == 'p1' and not os.environ.get('FEMO_NO_DIA')
    c0 = [es.p.vcycle_op_probe(m)[1] for m in PROBE_MODES] if has_dia else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        es.step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = es.launch_count() - l0 - (len(PROBE_MODES) if has_dia else 0)
    counts = [es.p.vcycle_op_probe(m)[1] - c0[m] - 1 for m in PROBE_MODES] if has_dia else None
    clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, es.outputs(), rank, world)
    kernels = time_kernels(es, counts, a.steps)
    step_info = dict(es.info)
    check = verify(es) if world == 1 else None
    es.info = step_info
    tt = torch.tensor([ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt.item())
    # one partitioned problem with `world` times the dofs: normalise to solves of the N=1 workload
    base_dofs = base_dofs_of(a.n, a.workload)
    norm = es.global_dofs / float(base_dofs) if world > 1 else 1.0
    value = norm * a.steps / (ms * 1e-3)

    # e2e: host buffers in, host buffers out, copies inside the timed region
    e2e = None
    if not a.no_e2e:
        import contextlib
        import io
        info = dict(es.info)
        if world == 1:
            # through the reference-facing API (FEA + FEAModel + Simulator, numpy in / numpy out)
            del es.vals, es.dv                  # the API path owns its own problem
            if a.workload != 'p1':
                es_nnz, es_N = es.nnz, es.p.N
                es.p = None                     # free the engine-level problem's arenas first
                es.u = es.f = es.dJdu = es.grad = es.lam = es.tmp = None
                torch.cuda.empty_cache()
            api = ApiStep(a.n, 2 if a.workload == 'p2' else 1)
            quiet = contextlib.redirect_stdout(io.StringIO())    # the reference prints "Converged reason" per solve
            quiet.__enter__()
            for _ in range(W):
                api.step()
            prob = api.fam.problem
            h0, d0 = prob.h2d_bytes, prob.d2h_bytes
            barrier()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                api.step()
            barrier()
            dt = time.perf_counter() - t0
            quiet.__exit__(None, None, None)
            h2d, d2h = (prob.h2d_bytes - h0) // a.steps, (prob.d2h_bytes - d0) // a.steps
            how = 'FEAModel + Simulator (numpy in/out; page-locked, version-tracked variable storage)'
            # the same chain with plain pageable, untracked numpy variables (what python_csdl_backend hands over)
            pageable = None
            if a.workload == 'p1':
                api = prob = None
                torch.cuda.empty_cache()
                api2 = ApiStep(a.n, 1, pinned=False)
                quiet = contextlib.redirect_stdout(io.StringIO())
                quiet.__enter__()
                for _ in range(W):
                    api2.step()
                prob2 = api2.fam.problem
                h0, d0 = prob2.h2d_bytes, prob2.d2h_bytes
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                for _ in range(a.steps):
                    api2.step()
                torch.cuda.synchronize()
                dt2 = time.perf_counter() - t1
                quiet.__exit__(None, None, None)
                pageable = dict(value=a.steps / dt2, unit=UNIT, ms_per_step=dt2 * 1e3 / a.steps,
                                h2d_bytes_per_step=int((prob2.h2d_bytes - h0) // a.steps),
                                d2h_bytes_per_step=int((prob2.d2h_bytes - d0) // a.steps),
                                path='FEAModel + Simulator with pageable, untracked numpy variables')
        else:
            # partitioned run: every rank feeds its slab of f from pinned host memory and reads back its
            # slab of the state, the gradient and J (the CSDL layer above is single-process in the reference)
            p = es.p
            hf = torch.full((p.M[0],), 0.1, dtype=torch.float64).pin_memory()
            hu = torch.empty(p.N, dtype=torch.float64).pin_memory()
            hg = torch.empty(p.M[0], dtype=torch.float64).pin_memory()

            def host_step():
                es.f.copy_(hf, non_blocking=True)
                J = es.step()
                hu.copy_(es.u, non_blocking=True)
                hg.copy_(es.grad, non_blocking=True)
                torch.cuda.synchronize()
                return J
            for _ in range(W):
                host_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                host_step()
            barrier()
            dt = time.perf_counter() - t0
            h2d, d2h = hf.numel() * 8 * world, (hu.numel() + hg.numel()) * 8 * world
            how = 'C-ABI step per rank with pinned host slabs of f (in), u and dJ/df (out)'
        td = torch.tensor([dt], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        dt = float(td.item())
        e2e = dict(value=norm * a.steps / dt, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                   ms_per_step=dt * 1e3 / a.steps, path=how)
        if world == 1 and pageable is not None:
            e2e['pageable'] = pageable
        es.info = info

    if rank == 0:
        peaks = {}
        pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        peak = float(peaks.get('hbm_gbs', 6650.0))
        # roofline of the instantiation with the largest share of the step (launches x duration, measured live)
        step_ms = ms / a.steps
        traffic = {}
        tp = os.path.join(ROOT, 'profiles', 'r02_kernel_traffic.json')
        if os.path.exists(tp) and a.workload == 'p1' and a.n == 4000 and world == 1:
            traffic = json.load(open(tp))
        for k in kernels:
            k['achieved_gbs'] = k['algorithmic_bytes'] / (k['launch_ms'] * 1e-3) / 1e9
            k['frac'] = k['achieved_gbs'] / peak
            k['share_of_step'] = k['launches_per_step'] * k['launch_ms'] / step_ms
            k['traffic'] = traffic.get(k['kernel'].split(' ')[0])
        dom = max((k for k in kernels if 'fp64-pipe bound' not in k['kernel']), key=lambda k: k['share_of_step'])
        out = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=W,
                   ms_per_step=ms / a.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64',
                   data='synthetic', config=arm_config(a.n, a.workload, world),
                   clocks=clocks, gpu_launches=int(launches), e2e=e2e,
                   roofline=dict(bound='hbm', kernel=dom['kernel'], achieved=dom['achieved_gbs'], peak=peak, unit='GB/s',
                                 frac=dom['frac'], traffic=dom['traffic'],
                                 traffic_source='profiles/r02_ncu_full_probe.csv (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch) -> profiles/r02_kernel_traffic.json',
                                 algorithmic_bytes=dom['algorithmic_bytes'], launch_ms=dom['launch_ms'],
                                 share_of_step=dom['share_of_step'],
                                 peak_source='MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks else 'fallback 6650 (of fallback)',
                                 kernels=kernels),
                   step_info=dict(es.info, verify=check, **({'amg_pattern_phase': es.setup} if a.workload == 'motor' else {})))
        if check is not None and not check['ok']:
            out['error'] = 'verification failed: %r' % (check,)
        if not a.no_cpu and world == 1:          # the CPU baseline is the N=1 workload: timed at N=1 only
            out['cpu_baseline'] = cpu_baseline(a.n)
            # same workload, two independent implementations: the functional must agree
            Jc, Jg = out['cpu_baseline']['J'], es.info.get('J')
            out['step_info']['J_cpu_port'] = Jc
            if Jg is not None and abs(Jg - Jc) > 1e-9 * abs(Jc):
                out['error'] = 'GPU and CPU-port functionals differ: %r vs %r' % (Jg, Jc)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
