"""Host-side mirror of the reference's operator interface for the hot path.

The names follow the two libraries the reference drives, so that parity tests
read like the reference's own call sequence (`F.cc` = FEniCSx driver, `M.cc` =
MFEM driver, `manual.py` = the UFL form file; paths relative to /root/reference):

  FEniCSx side (F.cc:679-688, 847-862)        here
  -----------------------------------------   ----------------------------------
  create_form(J) (coefficients d, E, u, nu)   ElasticityForm(mesh, E, nu, d, u)
  fem::petsc::create_matrix(*J_form)           create_matrix(form)
  DirichletBC bcl, bcr                         DirichletBC(marker, values)
  MatZeroEntries + assemble_matrix(set_block_  assemble_matrix(A, form, bcs)
    fn(A, ADD_VALUES), *J_form, {bcl, bcr})
    + set_diagonal(..., 1.) + MatAssembly
  ufcx tabulate_tensor(A, w, c, coord, ...)    tabulate_tensor(A, w, c, coordinate_dofs)
                                               tabulate_tensor_batched(form)
  MFEM side (M.cc:639, 1483-1546)
  damIntegrator::AssembleElementGrad           element_grad_batched(form)  (col-major, byNODES)
  AssembleElementVector / setF lambda          assemble_vector(A, form, f), apply_lifting(A, b, g, u)
  NewtonSolver (M.cc:1531-1549, F.cc:869-907)  NewtonSolver(form, bcs, f).solve()
  BilinearFormIntegrator::AssemblePA/AddMultPA PAOperator(form).AssemblePA()/AddMultPA()/Mult()
  damage smoothing (M.cc:1258-1315)            DamageSmoother(mesh).smooth(d, niter)
  strainTensor / stressTensor -> DG0 fields    cell_strain_stress(form)
    (M.cc:333-430,1551-1563; F.cc:909-942)
  CGSolver::SetRelTol/SetMaxIter/SetOperator/  CGSolver(...)
    SetPreconditioner/Mult                       (Jacobi instead of BoomerAMG: third party, out of scope)

Everything numerical runs in libfemb200.so (hand-written sm_100a CUDA) through
the C ABI of include/femb200.h; torch only owns device buffers and streams.
There is no CPU fallback: without a CUDA device every compute call raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _capi as capi
from .mesh import Mesh

_NP2T = {np.dtype(np.float64): torch.float64, np.dtype(np.int32): torch.int32, np.dtype(np.int64): torch.int64,
         np.dtype(np.uint8): torch.uint8}


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("femb200 needs a CUDA device (sm_100a): there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def to_device(a, dtype) -> torch.Tensor | None:
    """numpy (host) or torch (host/device) -> contiguous device tensor of `dtype`.
    Host arrays go through pinned memory with an asynchronous copy."""
    if a is None:
        return None
    dev = _require_cuda()
    tdt = _NP2T[np.dtype(dtype)]
    if isinstance(a, torch.Tensor):
        t = a
        if t.device.type != "cuda":
            t = t.contiguous().pin_memory().to(dev, non_blocking=True)
        return t.to(tdt).contiguous()
    h = torch.from_numpy(np.ascontiguousarray(a, dtype=dtype))
    return h.pin_memory().to(dev, non_blocking=True)


def _p(t: torch.Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


@dataclass
class DirichletBC:
    """Constrained dofs and their imposed values (F.cc:640,664).  `marker` is a
    per-dof uint8 array (global dof = 2 * node + component)."""
    marker: np.ndarray
    values: np.ndarray | None = None


def merge_bcs(bcs, ndofs: int):
    if bcs is None:
        return None
    if isinstance(bcs, DirichletBC):
        bcs = [bcs]
    if len(bcs) == 0:
        return None
    m = np.zeros(ndofs, dtype=np.uint8)
    for bc in bcs:
        mk = bc.marker.cpu().numpy() if isinstance(bc.marker, torch.Tensor) else np.asarray(bc.marker)
        m |= (mk != 0).astype(np.uint8)
    return m


class ElasticityForm:
    """The bilinear form J of the reference (manual.py:102) with its coefficients
    resident on the device: geometry, cell->dof maps, Young modulus per cell (DG0,
    manual.py:22), constant nu (manual.py:23), optional nodal damage d
    (manual.py:19) and current iterate u (manual.py:30)."""

    def __init__(self, mesh: Mesh, E, nu: float = 0.3, d=None, u=None, variant: int = capi.TANGENT_CLOSED):
        if mesh.etype == capi.Q1:
            raise ValueError("ElasticityForm: Q1 meshes are pattern only (coarse multigrid levels); there is no Q1 element")
        self.mesh = mesh
        self.etype, self.nnodes, self.ncells = mesh.etype, mesh.nnodes, mesh.ncells
        self.nd, self.nv = mesh.nd, mesh.nv
        self.nu = float(nu)
        self.variant = int(variant)
        self.x = to_device(mesh.x, np.float64)
        self.x_stride = int(mesh.x.shape[1])
        self.xdofmap = to_device(mesh.xdofmap, np.int32)
        self.dofmap = to_device(mesh.dofmap, np.int32)
        self.E = to_device(E, np.float64)
        self.d = to_device(d, np.float64)
        self.u = to_device(u, np.float64)
        if self.E.numel() != self.ncells:
            raise ValueError(f"E has {self.E.numel()} entries, expected one per cell ({self.ncells})")

    # coefficient updates between Newton iterations (host or device arrays)
    def set_u(self, u):
        self.u = to_device(u, np.float64)

    def set_damage(self, d):
        self.d = to_device(d, np.float64)

    def set_E(self, E):
        self.E = to_device(E, np.float64)

    def set_coordinates(self, x):
        self.x = to_device(x, np.float64)

    @property
    def geometry_vertices(self) -> np.ndarray:
        """Sorted node ids of the geometry vertices (the nodes xdofmap refers to)."""
        if getattr(self, "_gv", None) is None:
            self._gv = np.unique(np.asarray(self.mesh.xdofmap)).astype(np.int32)
            self._gv_dev = to_device(self._gv, np.int32)
        return self._gv

    def set_geometry(self, xv: torch.Tensor):
        """Refresh the coordinates of the geometry vertices only (role of mesh.geometry.x, which holds
        the P1 geometry, F.cc:213): xv is (len(geometry_vertices), x_stride) on the device or host."""
        gv = self.geometry_vertices
        xvd = xv if (isinstance(xv, torch.Tensor) and xv.is_cuda) else to_device(xv, np.float64)
        capi.call("femb200_scatter_rows", len(gv), self.x_stride, _p(self._gv_dev), _p(xvd), _p(self.x), _stream())


class Matrix:
    """CSR matrix in the dolfinx convention (rows in dof order, columns ascending,
    structural, bs = 2 expanded): rowptr int64, colidx int32, values float64, all
    on the device.  Owns the assembly plan (pattern + gather maps)."""

    def __init__(self, form: ElasticityForm):
        _require_cuda()
        self.form = form
        self._plan = C.c_void_p()
        capi.call("femb200_plan_create", form.etype, form.nnodes, form.ncells, _p(form.dofmap), _p(form.xdofmap),
                  _stream(), C.byref(self._plan))
        nn, nc, nnzb, nnz, bytes_ = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        mdeg = C.c_int32()
        capi.call("femb200_plan_sizes", self._plan, C.byref(nn), C.byref(nc), C.byref(nnzb), C.byref(nnz),
                  C.byref(mdeg), C.byref(bytes_))
        self.nnodes, self.ncells, self.nnz_blocks, self.nnz = nn.value, nc.value, nnzb.value, nnz.value
        self.max_block_degree, self.plan_bytes = mdeg.value, bytes_.value
        self.ndofs = 2 * self.nnodes
        self.values = torch.empty(self.nnz, dtype=torch.float64, device="cuda")
        self._rowptr = self._colidx = None
        self._bc_marker = None
        self.bc_dev = None

    def __del__(self):
        try:
            if getattr(self, "_plan", None) is not None and self._plan.value:
                capi.lib().femb200_plan_destroy(self._plan)
                self._plan = C.c_void_p()
        except Exception:
            pass

    @property
    def plan(self):
        return self._plan

    def _expand(self):
        self._rowptr = torch.empty(self.ndofs + 1, dtype=torch.int64, device="cuda")
        self._colidx = torch.empty(self.nnz, dtype=torch.int32, device="cuda")
        capi.call("femb200_plan_scalar_csr", self._plan, _p(self._rowptr), _p(self._colidx), _stream())

    @property
    def rowptr(self) -> torch.Tensor:
        if self._rowptr is None:
            self._expand()
        return self._rowptr

    @property
    def colidx(self) -> torch.Tensor:
        if self._colidx is None:
            self._expand()
        return self._colidx

    def block_csr(self):
        """(brp int64[nnodes+1], bcol int32[nnz_blocks]) device tensors (copies)."""
        brp = torch.empty(self.nnodes + 1, dtype=torch.int64, device="cuda")
        bcol = torch.empty(self.nnz_blocks, dtype=torch.int32, device="cuda")
        capi.call("femb200_plan_copy_block_csr", self._plan, _p(brp), _p(bcol), _stream())
        return brp, bcol

    def set_bcs(self, bcs):
        one = bcs[0] if isinstance(bcs, (list, tuple)) and len(bcs) == 1 else bcs
        if isinstance(one, DirichletBC) and isinstance(one.marker, torch.Tensor) and one.marker.is_cuda:
            # a single marker already on the device (large meshes): no round trip through the host
            self.bc_dev = (one.marker != 0).to(torch.uint8).contiguous()
            capi.call("femb200_plan_set_dirichlet", self._plan, _p(self.bc_dev), _stream())
            self._bc_marker = None
            return
        m = merge_bcs(bcs, self.ndofs)
        if m is None:
            capi.call("femb200_plan_set_dirichlet", self._plan, None, _stream())
            self.bc_dev = None
        else:
            self.bc_dev = to_device(m, np.uint8)
            capi.call("femb200_plan_set_dirichlet", self._plan, _p(self.bc_dev), _stream())
        self._bc_marker = m

    def set_option(self, key: str, value: int):
        """Kernel selection of the plan (femb200_plan_set_option): "assembly_path", "spmv_path", "spmv_cols", "spmv_compact"
        (0: PCG applies stream the compact values where the plan has them, 1: off), "vector_path", "prefetch_tiles",
        "stream_out", "damage_stage"."""
        capi.call("femb200_plan_set_option", self._plan, key.encode(), int(value))

    def get_option(self, key: str) -> int:
        """An option read back, or a read-only fact of the plan ("spmv_col_bits", "spmv_stencils", "spmv_compact_keys",
        "fast_records"): femb200_plan_get_option."""
        v = C.c_int()
        capi.call("femb200_plan_get_option", self._plan, key.encode(), C.byref(v))
        return v.value

    def mult_rows(self, x: torch.Tensor, y: torch.Tensor, lo: int, hi: int, dot: torch.Tensor | None = None,
                  accumulate: bool = False) -> torch.Tensor:
        """y = A x on the node rows [lo, hi) only (the rows a rank owns); `dot` (1 device double) gets <x, y>."""
        capi.call("femb200_spmv_rows", self._plan, _p(self.values), _p(x), _p(y), int(lo), int(hi), _p(dot),
                  int(accumulate), None, _stream())
        return y

    # --- operator interface (mfem::Operator::Mult / PETSc MatMult) -------------
    def mult(self, x: torch.Tensor, y: torch.Tensor | None = None) -> torch.Tensor:
        if y is None:
            y = torch.empty_like(x)
        capi.call("femb200_spmv", self._plan, _p(self.values), _p(x), _p(y), _stream())
        return y

    Mult = mult

    def diagonal(self) -> torch.Tensor:
        d = torch.empty(self.ndofs, dtype=torch.float64, device="cuda")
        capi.call("femb200_extract_diagonal", self._plan, _p(self.values), _p(d), _stream())
        return d

    def norms(self):
        """(Frobenius norm, trace), one 16-byte device->host read."""
        out = torch.empty(2, dtype=torch.float64, device="cuda")
        capi.call("femb200_matrix_norms", self._plan, _p(self.values), _p(out), _stream())
        f2, tr = out.cpu().tolist()
        return float(np.sqrt(f2)), float(tr)

    def to_scipy(self):
        import scipy.sparse as sp
        return sp.csr_matrix((self.values.cpu().numpy(), self.colidx.cpu().numpy(), self.rowptr.cpu().numpy()),
                             shape=(self.ndofs, self.ndofs))


def create_matrix(form: ElasticityForm) -> Matrix:
    """Role of dolfinx::fem::petsc::create_matrix(*J_form) (F.cc:688): builds the
    sparsity pattern once, on the device, from the cell->dof map alone."""
    return Matrix(form)


def assemble_matrix(A: Matrix, form: ElasticityForm | None = None, bcs=None, diag: float = 1.0,
                    norms_out: torch.Tensor | None = None) -> Matrix:
    """Role of the setJ lambda (F.cc:847-862): MatZeroEntries + assemble_matrix(
    set_block_fn(A, ADD_VALUES), J, bcs) + set_diagonal(..., 1.) + MatAssembly.
    One write-once gather kernel + (if any) the Dirichlet kernel.  `norms_out` (2 doubles on the
    device) receives (|K|_F^2, trace K) of the assembled matrix, fused into the same pass."""
    form = A.form if form is None else form
    if bcs is not None:
        A.set_bcs(bcs)
    if norms_out is not None:
        if diag != 1.0:
            raise ValueError("norms_out needs the unit Dirichlet diagonal")
        capi.call("femb200_assemble_matrix_norms", A.plan, _p(form.x), form.x_stride, _p(form.E), form.nu, _p(form.d),
                  _p(form.u), form.variant, _p(A.values), _p(norms_out), _stream())
        return A
    capi.call("femb200_assemble_matrix", A.plan, _p(form.x), form.x_stride, _p(form.E), form.nu, _p(form.d),
              _p(form.u), form.variant, _p(A.values), _stream())
    if diag != 1.0 and A.bc_dev is not None:
        capi.call("femb200_apply_dirichlet", A.plan, _p(A.values), float(diag), _stream())
    return A


def assemble_matrix_nobc(A: Matrix, form: ElasticityForm | None = None) -> Matrix:
    """The unconstrained tangent (no Dirichlet rows/cols): what apply_lifting needs."""
    form = A.form if form is None else form
    capi.call("femb200_assemble_matrix_nobc", A.plan, _p(form.x), form.x_stride, _p(form.E), form.nu, _p(form.d),
              _p(form.u), form.variant, _p(A.values), _stream())
    return A


def assemble_vector(A: Matrix, form: ElasticityForm | None = None, f=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """Role of assemble_vector(F) (F.cc:825) / ParNonlinearForm::Mult -> AssembleElementVector
    (M.cc:559-637): b = F(u) = int sigma(u):eps(v) - int f.v, no boundary treatment.  `f` is the
    nodal body force (nnodes x 2, host or device) or None; the current iterate is form.u."""
    form = A.form if form is None else form
    if form.u is None:
        form.set_u(np.zeros(2 * form.nnodes))
    fd = to_device(f, np.float64)
    if out is None:
        out = torch.empty(2 * form.nnodes, dtype=torch.float64, device="cuda")
    capi.call("femb200_assemble_vector", A.plan, _p(form.x), form.x_stride, _p(form.E), form.nu, _p(form.d),
              _p(form.u), _p(fd), _p(out), _stream())
    return out


def apply_lifting(A: Matrix, b: torch.Tensor, g: torch.Tensor, u: torch.Tensor, scale: float = -1.0) -> torch.Tensor:
    """apply_lifting(b, {J}, {bcs}, {u}, scale) + set_bc(b, bcs, u, scale) of the setF lambda
    (F.cc:826-836): b -= scale * J[:, bc] (g - u)_bc on the free dofs, b[bc] = scale * (g - u)[bc].
    A.values must hold the UNCONSTRAINED tangent (assemble_matrix_nobc)."""
    capi.call("femb200_apply_lifting", A.plan, _p(A.values), _p(g), _p(u), float(scale), _p(b), None, _stream())
    return b


class NewtonSolver:
    """The Newton loop around the hot path (mfem::NewtonSolver, M.cc:1531-1549; dolfinx nls::petsc::NewtonSolver,
    F.cc:705-714,869-907).  Per iteration: residual b = F(u) with the Dirichlet lifting (setF, F.cc:817-845), tangent
    J(u) with Dirichlet rows/columns (setJ, F.cc:847-862), Jacobi-PCG solve J du = b, u <- u - du.
    preconditioner="mg" solves with multigrid-PCG instead (MultigridPreconditioner on `hierarchy`, set up again for
    every tangent; one GPU only, no `part`).

    Both convergence conventions of the reference (doc.tex:2065-2068):
      convention="mfem"     |b| <= max(rel_tol |b_0|, abs_tol), b_0 = the first residual (M.cc:1535-1541);
      convention="dolfinx"  |b| / r_0 < rel_tol or |b| < abs_tol with r_0 = |du_0|, the norm of the FIRST
                            SOLUTION INCREMENT (set after the first update; before it only the absolute test
                            can stop the loop) -- the reason FEniCSx iterates twice more than MFEM.
    `part` (a dist.StripPartition) runs the same loop on one partition per rank: owned-row norms are all-reduced,
    u gets its ghost update after every increment (newton_solver.set_form, F.cc:865-866) and the linear solve is
    femb200_dist_pcg; without it the solver works on the whole mesh (a one-rank partition).
    The tangent is assembled only when an increment is actually computed (after the convergence test), and once
    u carries the boundary values (every iteration after the first) the lifting reduces to set_bc."""

    mg = None   # MultigridPreconditioner with preconditioner="mg"

    def __init__(self, form: ElasticityForm, bcs, f=None, rel_tol=1e-7, abs_tol=5e-8, max_iter=10, cg_rel_tol=1e-12,
                 cg_max_iter=2000, convention: str = "mfem", part=None, transport: str = "auto", group=None,
                 preconditioner: str = "jacobi", hierarchy=None):
        from . import dist
        if convention not in ("mfem", "dolfinx"):
            raise ValueError("convention must be 'mfem' or 'dolfinx'")
        if preconditioner not in ("jacobi", "mg"):
            raise ValueError("preconditioner must be 'jacobi' or 'mg'")
        if preconditioner == "mg" and part is not None:
            raise ValueError("the multigrid preconditioner runs on one GPU: it cannot be combined with part=")
        if preconditioner == "mg" and hierarchy is None:
            raise ValueError('preconditioner="mg" needs hierarchy= (mesh.lattice_hierarchy / refine_uniform_hierarchy)')
        self.form, self.f = form, to_device(f, np.float64)
        self.rel_tol, self.abs_tol, self.max_iter, self.convention = rel_tol, abs_tol, max_iter, convention
        self.A = create_matrix(form)
        self.A.set_bcs(bcs)
        one = bcs[0] if isinstance(bcs, (list, tuple)) and len(bcs) == 1 else bcs
        if isinstance(one, DirichletBC) and isinstance(one.values, torch.Tensor) and one.values.is_cuda:
            self.g = one.values.to(torch.float64).contiguous()
        else:
            gv = np.zeros(self.A.ndofs)
            for bc in ([bcs] if isinstance(bcs, DirichletBC) else bcs):
                if bc.values is not None:
                    m = np.asarray(bc.marker) != 0
                    gv[m] = np.asarray(bc.values)[m]
            self.g = to_device(gv, np.float64)
        self.part = dist.trivial_partition(form.mesh) if part is None else part
        self.cg = dist.DistCG(self.A, self.part, rel_tol=cg_rel_tol, max_iter=cg_max_iter, jacobi=False,
                              transport=transport, group=group)
        self.cg_rel_tol, self.cg_max_iter = cg_rel_tol, cg_max_iter
        self.mg = MultigridPreconditioner(self.A, hierarchy) if preconditioner == "mg" else None
        self._lo, self._hi = 2 * self.part.own_lo, 2 * self.part.own_hi
        self._b = torch.empty(self.A.ndofs, dtype=torch.float64, device="cuda")
        self._du = torch.zeros(self.A.ndofs, dtype=torch.float64, device="cuda")
        self._nrm = torch.zeros(1, dtype=torch.float64, device="cuda")
        self._lifted = False          # does u carry the boundary values already?
        self._tangent_ready = False   # A.values holds the unconstrained tangent of the current u
        self.residual_norms, self.linear_iterations, self.linear_converged = [], [], []

    def close(self):
        if self.mg is not None:
            self.mg.close()
        self.cg.close()

    # -- building blocks (one Newton linearisation = residual() + increment()) -----------------
    def prepare_tangent(self) -> bool:
        """Assembles the unconstrained tangent ahead of residual() when it does not depend on the iterate (a form
        without damage: J is the linear stiffness, M.cc:873-881), e.g. while u is still on its way to the device;
        returns False (and does nothing) for a form whose tangent needs u."""
        if self.form.d is not None:
            return False
        assemble_matrix_nobc(self.A, self.form)
        self._tangent_ready = True
        return True

    def residual(self, u: torch.Tensor) -> torch.Tensor:
        """b = F(u) with apply_lifting + set_bc (scale -1), setF lambda F.cc:817-845."""
        form, A, b = self.form, self.A, self._b
        form.u = u
        assemble_vector(A, form, self.f, out=b)
        if form.d is not None:
            self._tangent_ready = False     # the tangent of a damaged form depends on u
        if self._lifted:
            capi.call("femb200_set_bc", A.plan, _p(self.g), _p(u), -1.0, _p(b), _stream())
        else:
            if not self._tangent_ready:
                assemble_matrix_nobc(A, form)
                self._tangent_ready = True
            capi.call("femb200_apply_lifting", A.plan, _p(A.values), _p(self.g), _p(u), -1.0, _p(b), None, _stream())
        return b

    def norm(self, v: torch.Tensor) -> float:
        """l2 norm over the owned dofs of every rank (one 8-byte read back: the convergence decision is the host's)."""
        n = self._hi - self._lo
        off = C.c_void_p(v.data_ptr() + 8 * self._lo)
        capi.call("femb200_dot", n, off, off, _p(self._nrm), _stream())
        self.cg.op.allreduce_sum(self._nrm)
        return float(np.sqrt(self._nrm.item()))

    def increment(self, b: torch.Tensor, fixed_iters: int = 0) -> torch.Tensor:
        """du = J(u)^-1 b: tangent with Dirichlet rows/columns (setJ lambda F.cc:847-862) + Jacobi-PCG."""
        form, A = self.form, self.A
        if self._tangent_ready:
            capi.call("femb200_apply_dirichlet", A.plan, _p(A.values), 1.0, _stream())
        else:
            assemble_matrix(A, form)
        self._tangent_ready = False
        if self.mg is not None:
            if fixed_iters:
                raise ValueError("fixed_iters is not supported with the multigrid preconditioner")
            self.mg.setup()     # Galerkin levels, smoother and coarse inverse of the new tangent
            it, _, conv = self.mg.solve(b, self._du, self.cg_rel_tol, 0.0, self.cg_max_iter)
            self.linear_iterations.append(it)
            self.linear_converged.append(conv)
            return self._du
        self.cg.update_preconditioner()
        self.cg.solve(b, self._du, fixed_iters=fixed_iters)
        self.linear_iterations.append(self.cg.iterations)
        if hasattr(self, "linear_converged"):   # absent on solvers assembled with __new__ (bench.py's end-to-end leg)
            self.linear_converged.append(self.cg.converged)
        return self._du

    def update(self, u: torch.Tensor, du: torch.Tensor) -> torch.Tensor:
        """u <- u - du on the owned dofs, then the ghost update of u (F.cc:865-866)."""
        n = self._hi - self._lo
        capi.call("femb200_axpy", n, -1.0, C.c_void_p(du.data_ptr() + 8 * self._lo), C.c_void_p(u.data_ptr() + 8 * self._lo),
                  _stream())
        self.cg.op.halo(u)
        self._lifted = True
        return u

    def solve(self, u0=None) -> torch.Tensor:
        A = self.A
        u = torch.zeros(A.ndofs, dtype=torch.float64, device="cuda") if u0 is None else to_device(u0, np.float64).clone()
        self.residual_norms, self.linear_iterations, self.increment_norms = [], [], []
        self.linear_converged = []
        self._lifted = False
        self.converged = False
        r0 = None
        for it in range(self.max_iter + 1):
            nrm = self.norm(self.residual(u))
            self.residual_norms.append(nrm)
            if self.convention == "mfem":
                self.converged = nrm <= max(self.rel_tol * self.residual_norms[0], self.abs_tol)
            else:
                self.converged = nrm < self.abs_tol or (r0 is not None and nrm / r0 < self.rel_tol)
            if self.converged or it == self.max_iter:
                break
            du = self.increment(self._b)
            if it == 0:
                r0 = self.norm(du)
            self.increment_norms.append(r0 if it == 0 else None)
            self.update(u, du)
        self.iterations = len(self.residual_norms) - 1
        return u


def tabulate_tensor_batched(form: ElasticityForm, layout: int = capi.ROWMAJOR_INTERLEAVED,
                            out: torch.Tensor | None = None) -> torch.Tensor:
    """All element tangents in one launch: ncells x (2 nd)^2, ufcx layout
    (row-major, interleaved dofs) by default."""
    _require_cuda()
    n = 2 * form.nd
    if out is None:
        out = torch.empty((form.ncells, n, n), dtype=torch.float64, device="cuda")
    capi.call("femb200_tabulate_tensor_batched", form.etype, form.ncells, _p(out), _p(form.x), form.x_stride,
              _p(form.xdofmap), _p(form.dofmap), _p(form.E), form.nu, _p(form.d), _p(form.u), form.variant,
              int(layout), _stream())
    return out


def element_grad_batched(form: ElasticityForm) -> torch.Tensor:
    """damIntegrator::AssembleElementGrad for every element (M.cc:639-916):
    elmat column-major, dofs byNODES.  Returned so that out[e, c, r] = elmat(r, c),
    i.e. out[e].T is the DenseMatrix."""
    return tabulate_tensor_batched(form, capi.COLMAJOR_BYNODES)


def tabulate_tensor(A: np.ndarray, w: np.ndarray, c: np.ndarray, coordinate_dofs: np.ndarray,
                    entity_local_index=None, quadrature_permutation=None) -> None:
    """Host shim with the ufcx signature for the P1 form J (batch of one cell):
    `A` (6x6 row-major, interleaved dofs) is caller-owned and ACCUMULATED into,
    as ffcx kernels do.  w = [d0,d1,d2, E, u0x,u0y,u1x,u1y,u2x,u2y] (coefficient
    order of manual.py:19,22,30), c = [nu] (manual.py:23), coordinate_dofs 3x3
    (xyz-padded, F.cc:213)."""
    from .mesh import P1
    cd = np.asarray(coordinate_dofs, dtype=np.float64).reshape(3, 3)
    w = np.asarray(w, dtype=np.float64).ravel()
    m = Mesh(P1, cd.copy(), np.array([[0, 1, 2]], dtype=np.int32), np.array([[0, 1, 2]], dtype=np.int32))
    d = w[0:3] if np.any(w[0:3] != 0.0) else None
    form = ElasticityForm(m, w[3:4], float(np.asarray(c).ravel()[0]), d=d, u=w[4:10])
    Ae = tabulate_tensor_batched(form).cpu().numpy().reshape(-1)
    Av = np.asarray(A).reshape(-1)
    Av += Ae


class DamageSmoother:
    """The reference's damage-field smoothing over the vertex graph of the triangulation
    (M.cc:1209-1315; the Python driver builds a SciPy adjacency matrix for it, F.py:160-199):
    niter double sweeps d_l = max(sum over edge neighbours / edge count, d_l), the first of each
    pair only where d_l < 0.01.  The graph is the block pattern of a P1 plan on the geometry
    vertices, built once on the device; `d` is indexed by node id like ElasticityForm.d."""

    def __init__(self, mesh: Mesh):
        _require_cuda()
        if mesh.nv != 3:
            raise ValueError("damage smoothing is defined on triangulations (the reference has no quads)")
        self.nnodes = mesh.nnodes
        self._tri = to_device(mesh.xdofmap, np.int32)
        self._plan = C.c_void_p()
        capi.call("femb200_plan_create", capi.P1, mesh.nnodes, mesh.ncells, _p(self._tri), _p(self._tri), _stream(),
                  C.byref(self._plan))
        self._work = torch.empty(self.nnodes, dtype=torch.float64, device="cuda")

    def __del__(self):
        try:
            if getattr(self, "_plan", None) is not None and self._plan.value:
                capi.lib().femb200_plan_destroy(self._plan)
                self._plan = C.c_void_p()
        except Exception:
            pass

    def smooth(self, d, niter: int = 8, threshold: float = 0.01) -> torch.Tensor:
        """niter = 8 * (max_refine + 1) in the reference (M.cc:1258).  Returns a new device tensor."""
        dd = to_device(d, np.float64).clone()
        if dd.numel() != self.nnodes:
            raise ValueError(f"d has {dd.numel()} entries, expected one per node ({self.nnodes})")
        capi.call("femb200_smooth_damage", self._plan, _p(dd), _p(self._work), int(niter), float(threshold), _stream())
        return dd


def cell_strain_stress(form: ElasticityForm, stress: bool = True):
    """DG0 output fields of the reference (strainTensor / stressTensor projected on a 3-component
    DG0 space, M.cc:333-430,1551-1563; strain/stress expressions interpolated into S, F.cc:909-942):
    (ncells, 3) device tensors (xx, xy, yy) evaluated at the cell centroid for the current form.u."""
    if form.u is None:
        raise ValueError("form.u (the displacement) is not set")
    eps = torch.empty((form.ncells, 3), dtype=torch.float64, device="cuda")
    sig = torch.empty((form.ncells, 3), dtype=torch.float64, device="cuda") if stress else None
    capi.call("femb200_cell_strain_stress", form.etype, form.ncells, _p(form.xdofmap), _p(form.dofmap), _p(form.x),
              form.x_stride, _p(form.E), form.nu, _p(form.d), _p(form.u), _p(eps), _p(sig), _stream())
    return eps, sig


class PAOperator:
    """Partial-assembly (matrix-free) operator: the AssemblePA / AddMultPA /
    AssembleDiagonalPA role of an mfem BilinearFormIntegrator."""

    def __init__(self, form: ElasticityForm, bcs=None, diag: float = 1.0):
        _require_cuda()
        self.form = form
        self.ndofs = 2 * form.nnodes
        self._pa = C.c_void_p()
        self._bcs, self._diag = bcs, float(diag)
        self.bc_dev = None
        self.generation = 0   # counts the AssemblePA calls: each one replaces the device operator behind `handle`
        self.AssemblePA()

    def AssemblePA(self):
        f = self.form
        self.generation += 1
        if self._pa.value:
            capi.lib().femb200_pa_destroy(self._pa)
            self._pa = C.c_void_p()
        capi.call("femb200_pa_create", f.etype, f.nnodes, f.ncells, _p(f.dofmap), _p(f.xdofmap), _p(f.x), f.x_stride,
                  _p(f.E), f.nu, _stream(), C.byref(self._pa))
        m = merge_bcs(self._bcs, self.ndofs)
        if m is not None:
            self.bc_dev = to_device(m, np.uint8)
            capi.call("femb200_pa_set_dirichlet", self._pa, _p(self.bc_dev), self._diag, _stream())

    def __del__(self):
        try:
            if getattr(self, "_pa", None) is not None and self._pa.value:
                capi.lib().femb200_pa_destroy(self._pa)
                self._pa = C.c_void_p()
        except Exception:
            pass

    @property
    def handle(self):
        return self._pa

    def mult(self, x: torch.Tensor, y: torch.Tensor | None = None) -> torch.Tensor:
        if y is None:
            y = torch.empty_like(x)
        capi.call("femb200_pa_apply", self._pa, _p(x), _p(y), _stream())
        return y

    Mult = mult

    def AddMultPA(self, x: torch.Tensor, y: torch.Tensor) -> None:
        """y += A x (mfem AddMultPA semantics)."""
        if getattr(self, "_work", None) is None:
            self._work = torch.empty(self.ndofs, dtype=torch.float64, device="cuda")
        capi.call("femb200_add_mult_pa", self._pa, self.ndofs, _p(x), _p(y), _p(self._work), _stream())

    def diagonal(self) -> torch.Tensor:
        d = torch.empty(self.ndofs, dtype=torch.float64, device="cuda")
        capi.call("femb200_pa_diagonal", self._pa, _p(d), _stream())
        return d

    AssembleDiagonalPA = diagonal


class MultigridPreconditioner:
    """Geometric multigrid V-cycle for an operator `A` with its Dirichlet conditions set -- an assembled Matrix (P1, P2,
    Q2) or a matrix-free PAOperator (P2, Q2) -- on a nested MeshHierarchy whose finest mesh is A's mesh
    (mesh.lattice_hierarchy, mesh.quad_lattice_hierarchy, mesh.refine_uniform_hierarchy).

    Levels: A itself, then the Galerkin operators P^T A P of the coarser meshes, computed on the device by
    femb200_mg_setup; the hierarchy is cut at the first level with at most `coarse_max` dofs, whose dense inverse
    (torch.linalg on the device) is the coarse solve.  For a PAOperator the first step must be a p-coarsening (P2 -> P1,
    Q2 -> Q1 on the same cells): its Galerkin operator is summed from the operator's per-cell data, the fine matrix is
    never assembled.  Smoother: Chebyshev of `degree` on D^-1 A over [lo_frac lambda, lambda], the same before and after
    the coarse correction, so the V-cycle is symmetric positive definite.  Call setup() after every reassembly of
    A.values (the V-cycle reads A.values in place) or of the PAOperator: PAOperator.AssemblePA replaces the device
    operator, so setup() then rebuilds the device handle on the new one, and apply() / solve() refuse to run until it has."""

    def __init__(self, A, hierarchy, degree: int = 2, coarse_max: int = 4096, lo_frac: float = 0.25):
        from .mesh import P1, P2, Q1, Q2, ELEM_NAME
        _require_cuda()
        if not isinstance(A, (Matrix, PAOperator)):
            raise ValueError("the multigrid preconditioner needs a Matrix or a PAOperator")
        self.matrix_free = isinstance(A, PAOperator)
        fine = hierarchy.meshes[-1]
        mine = A.form.mesh
        same = fine is mine or (fine.ndofs == A.ndofs and fine.etype == A.form.etype and fine.ncells == mine.ncells and
                                np.array_equal(fine.dofmap, mine.dofmap) and np.array_equal(fine.x, mine.x))
        if not same:
            raise ValueError(f"the finest mesh of the hierarchy ({fine.ndofs} dofs) is not the mesh of the operator "
                             f"({A.ndofs} dofs)")
        nlev = len(hierarchy.meshes)
        sizes = [m.ndofs for m in hierarchy.meshes]
        if nlev < 2:
            raise ValueError("the hierarchy has no mesh coarser than the fine one")
        widths = {int(np.asarray(t).shape[1]) for t in hierarchy.maps}
        if len(widths) != 1 or not widths <= {2, 4}:
            raise ValueError(f"the transfer maps must all have width 2 or all width 4, got widths {sorted(widths)}")
        self.width = widths.pop()
        coarse_type = P1 if self.width == 2 else Q1
        for m in hierarchy.meshes[:-1]:
            if m.etype != coarse_type:
                raise ValueError(f"coarse levels must be {ELEM_NAME[coarse_type]} for transfer maps of width "
                                 f"{self.width}, got {ELEM_NAME.get(m.etype, m.etype)}")
        if self.matrix_free:
            first = hierarchy.meshes[-2]
            want = {P2: P1, Q2: Q1}.get(fine.etype)
            if want is None or first.etype != want or first.ncells != fine.ncells:
                raise ValueError("a matrix-free (PAOperator) fine level needs a P2 or Q2 mesh whose first coarsening is a "
                                 "p-coarsening (P2 -> P1 or Q2 -> Q1 on the same cells)")
        keep = next((k for k in range(nlev - 2, -1, -1) if sizes[k] <= coarse_max), None)
        if keep is None:
            raise ValueError(f"the coarsest mesh of the hierarchy has {sizes[0]} dofs, more than coarse_max = {coarse_max}")
        self.A, self.degree, self.coarse_max = A, int(degree), int(coarse_max)
        meshes = hierarchy.meshes[keep:]           # coarsest first
        maps = hierarchy.maps[keep:]
        fine_marker = A.bc_dev.cpu().numpy() if A.bc_dev is not None else np.zeros(A.ndofs, np.uint8)
        markers = type(hierarchy)(meshes, maps).markers(fine_marker)
        # level l = 0 (fine) .. L (coarsest)
        self.nlevels = len(meshes) - 1
        self._keep = []                            # device arrays the plans and the handle borrow
        self._plans = []
        for k in range(self.nlevels - 1, -1, -1):  # coarse levels 1 .. L
            m = meshes[k]
            dm = to_device(m.dofmap, np.int32)
            plan = C.c_void_p()
            capi.call("femb200_plan_create", m.etype, m.nnodes, m.ncells, _p(dm), _p(dm), _stream(), C.byref(plan))
            self._plans.append(plan)
            self._keep.append(dm)
        dmaps = [to_device(maps[k], np.int32) for k in range(self.nlevels - 1, -1, -1)]
        dbcs = [to_device(markers[k], np.uint8) for k in range(self.nlevels - 1, -1, -1)]
        self._keep += dmaps + dbcs
        self._dmaps, self._dbcs, self._lo_frac = dmaps, dbcs, float(lo_frac)
        self._handle = C.c_void_p()
        self._create()
        self.level_meshes = list(reversed(meshes))  # fine first
        self._work = None
        self.ready = False

    def _create(self):
        """The device handle on the operator as it is now (it borrows the operator, the plans, maps and markers)."""
        arr = lambda ts: (C.c_void_p * len(ts))(*[t.value if isinstance(t, C.c_void_p) else t.data_ptr() for t in ts])
        kind, op = (capi.OP_PA, self.A.handle) if self.matrix_free else (capi.OP_CSR, self.A.plan)
        capi.call("femb200_mg_create_op", kind, op, self.nlevels, arr(self._plans), arr(self._dmaps), self.width,
                  arr(self._dbcs), self.degree, self._lo_frac, _stream(), C.byref(self._handle))
        self._generation = getattr(self.A, "generation", 0)

    def _sync_operator(self):
        """After PAOperator.AssemblePA the handle points at a freed operator: build it again on the new one."""
        if self.matrix_free and self.A.generation != self._generation:
            self.ready = False
            capi.lib().femb200_mg_destroy(self._handle)
            self._handle = C.c_void_p()
            self._create()

    def _check_ready(self, what: str):
        if self.matrix_free and self.A.generation != self._generation:
            raise RuntimeError(f"MultigridPreconditioner.{what}: the PAOperator was reassembled (AssemblePA); "
                               "call setup() first")
        if not self.ready:
            raise RuntimeError(f"MultigridPreconditioner.{what}: call setup() first")

    def _fine_values(self):
        return None if self.matrix_free else _p(self.A.values)

    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle.value:
            capi.lib().femb200_mg_destroy(self._handle)
            self._handle = C.c_void_p()
        for p in getattr(self, "_plans", []):
            if p.value:
                capi.lib().femb200_plan_destroy(p)
        self._plans = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._handle

    def sizes(self):
        """(dofs per level, nnz per level, lambda per level, device bytes of the handle), fine level first."""
        L = self.nlevels
        nl = C.c_int()
        nd, nz, lam = (C.c_int64 * (L + 1))(), (C.c_int64 * (L + 1))(), (C.c_double * (L + 1))()
        by = C.c_int64()
        capi.call("femb200_mg_sizes", self._handle, C.byref(nl), nd, nz, lam, C.byref(by))
        return list(nd), list(nz), list(lam), by.value

    @property
    def lambdas(self):
        return self.sizes()[2]

    def galerkin(self, level: int):
        """Recompute A_{level+1} = P^T A_level P alone (timing and tests; setup() runs every level).  Level 0 of a
        matrix-free operator is the element Galerkin step."""
        self._sync_operator()
        capi.call("femb200_mg_galerkin", self._handle, self._fine_values() if level == 0 else None, int(level), _stream())

    def setup(self):
        """Numeric phase: Galerkin cascade, smoother set-up (D^-1, lambda) and the coarse inverse."""
        self._sync_operator()
        capi.call("femb200_mg_setup", self._handle, self._fine_values(), _stream())
        self.set_coarse_inverse()

    def set_coarse_inverse(self):
        Ac = self.coarse_matrix()
        inv = torch.linalg.inv(Ac)
        inv = (0.5 * (inv + inv.T)).contiguous()   # exactly symmetric: keeps the V-cycle symmetric
        capi.call("femb200_mg_set_coarse_inverse", self._handle, _p(inv), _stream())
        self.ready = True

    def coarse_matrix(self) -> torch.Tensor:
        n = self.sizes()[0][-1]
        out = torch.empty((n, n), dtype=torch.float64, device="cuda")
        capi.call("femb200_mg_coarse_matrix", self._handle, _p(out), _stream())
        return out

    def level_values(self, level: int) -> torch.Tensor:
        """CSR values of level 1..L in the pattern of that level's P1 / Q1 plan (level_csr)."""
        out = torch.empty(self.sizes()[1][level], dtype=torch.float64, device="cuda")
        capi.call("femb200_mg_level_values", self._handle, int(level), _p(out), _stream())
        return out

    def level_csr(self, level: int):
        """(rowptr int64, colidx int32) device tensors of the scalar CSR pattern of level 1..L."""
        n = self.sizes()[0][level]
        nnz = self.sizes()[1][level]
        rp = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        ci = torch.empty(nnz, dtype=torch.int32, device="cuda")
        capi.call("femb200_plan_scalar_csr", self._plans[level - 1], _p(rp), _p(ci), _stream())
        return rp, ci

    def restrict(self, level: int, b: torch.Tensor, t: torch.Tensor | None = None) -> torch.Tensor:
        """P^T (b - t) from `level` to level + 1 (t = A x, or None for x = 0)."""
        out = torch.empty(self.sizes()[0][level + 1], dtype=torch.float64, device="cuda")
        self._sync_operator()
        capi.call("femb200_mg_restrict", self._handle, int(level), _p(b), _p(t), _p(out), _stream())
        return out

    def prolong(self, level: int, xc: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        """x += P xc from level + 1 to `level` (in place)."""
        self._sync_operator()
        capi.call("femb200_mg_prolong", self._handle, int(level), _p(xc), _p(x), _stream())
        return x

    def apply(self, r: torch.Tensor, z: torch.Tensor | None = None) -> torch.Tensor:
        """z = B r: one V-cycle."""
        self._check_ready("apply")
        if z is None:
            z = torch.empty_like(r)
        elif z.data_ptr() == r.data_ptr():
            raise ValueError("MultigridPreconditioner.apply: z must not alias r (the V-cycle reads r after writing z)")
        capi.call("femb200_mg_vcycle", self._handle, _p(r), _p(z), _stream())
        return z

    Mult = apply

    def apply_timed(self, r: torch.Tensor, z: torch.Tensor) -> np.ndarray:
        """One V-cycle with a CUDA event after every launch: (levels, 5) milliseconds per level of its SpMVs,
        Chebyshev vector passes, restriction, prolongation and coarse GEMV (femb200_mg_vcycle_timed)."""
        self._check_ready("apply_timed")
        if z.data_ptr() == r.data_ptr():
            raise ValueError("MultigridPreconditioner.apply_timed: z must not alias r")
        ms = np.zeros((self.nlevels + 1) * 5)
        capi.call("femb200_mg_vcycle_timed", self._handle, _p(r), _p(z), ms.ctypes.data_as(C.c_void_p), _stream())
        return ms.reshape(self.nlevels + 1, 5)

    def solve(self, b: torch.Tensor, x: torch.Tensor, rel_tol: float = 1e-12, abs_tol: float = 0.0, max_iter: int = 2000,
              check_every: int = 1):
        """PCG on A with this preconditioner (femb200_pcg_mg): returns (iterations, final <B r, r>^1/2, converged)."""
        self._check_ready("solve")
        n = self.A.ndofs
        if self._work is None or self._work.numel() < 4 * n + 64:
            self._work = torch.empty(4 * n + 64, dtype=torch.float64, device="cuda")
        it, fn, cv = C.c_int(), C.c_double(), C.c_int()
        capi.call("femb200_pcg_mg", self._handle, _p(b), _p(x), float(rel_tol), float(abs_tol), int(max_iter),
                  int(check_every), _p(self._work), C.byref(it), C.byref(fn), C.byref(cv), _stream())
        return it.value, fn.value, bool(cv.value)


class CGSolver:
    """mfem::CGSolver surface (M.cc:1502,1525-1528): SetRelTol / SetAbsTol /
    SetMaxIter / SetOperator / SetPreconditioner / Mult, zero initial guess
    (iterative_mode = false).  The preconditioner is Jacobi, none, or geometric multigrid
    (SetPreconditioner("mg", hierarchy=...) or a MultigridPreconditioner)."""

    def __init__(self, rel_tol: float = 1e-12, abs_tol: float = 0.0, max_iter: int = 2000, check_every: int | None = None):
        """check_every: iterations between host convergence polls; None = 25 for Jacobi / none, 1 for multigrid
        (a V-cycle queued after convergence is wasted work, a poll costs one synchronisation)."""
        self.rel_tol, self.abs_tol, self.max_iter = rel_tol, abs_tol, max_iter
        self.check_every = check_every
        self.op = None
        self.dinv = None
        self.mg = None
        self._work = None
        self.iterations, self.final_norm, self.converged = 0, 0.0, False

    def SetRelTol(self, v):
        self.rel_tol = float(v)

    def SetAbsTol(self, v):
        self.abs_tol = float(v)

    def SetMaxIter(self, v):
        self.max_iter = int(v)

    def SetOperator(self, op):
        self.op = op
        self.dinv = None
        self.mg = None

    def SetPreconditioner(self, kind="jacobi", hierarchy=None, **mg_options):
        """"jacobi", "none" / None, "mg" (geometric multigrid on `hierarchy`, set up now; call its setup() again
        after reassembling the operator), or a MultigridPreconditioner of the operator."""
        self.mg = None
        if isinstance(kind, MultigridPreconditioner):
            if kind.A is not self.op:
                raise ValueError("the multigrid preconditioner was built for another operator")
            self.dinv, self.mg = None, kind
            return
        if kind is None or kind == "none":
            self.dinv = None
            return
        if kind == "mg":
            if not isinstance(self.op, (Matrix, PAOperator)):
                raise ValueError("the multigrid preconditioner needs a Matrix or a PAOperator")
            if hierarchy is None:
                raise ValueError('SetPreconditioner("mg") needs hierarchy= (mesh.lattice_hierarchy / quad_lattice_hierarchy / '
                                 'refine_uniform_hierarchy)')
            self.dinv = None
            self.mg = MultigridPreconditioner(self.op, hierarchy, **mg_options)
            self.mg.setup()
            return
        if kind != "jacobi":
            raise ValueError(f"unknown preconditioner {kind!r}: 'jacobi', 'mg' or 'none'")
        diag = self.op.diagonal()
        self.dinv = torch.empty_like(diag)
        capi.call("femb200_jacobi_setup", diag.numel(), _p(diag), _p(self.dinv), _stream())

    def GetNumIterations(self):
        return self.iterations

    def GetConverged(self):
        return self.converged

    def GetFinalNorm(self):
        return self.final_norm

    def Mult(self, b: torch.Tensor, x: torch.Tensor | None = None, fixed_iters: int = 0) -> torch.Tensor:
        if self.op is None:
            raise RuntimeError("CGSolver.Mult: SetOperator first")
        n = b.numel()
        if x is None:
            x = torch.empty_like(b)
        if self.mg is not None:
            if fixed_iters:
                raise ValueError("fixed_iters is not supported with the multigrid preconditioner")
            self.iterations, self.final_norm, self.converged = self.mg.solve(
                b, x, self.rel_tol, self.abs_tol, self.max_iter, 1 if self.check_every is None else self.check_every)
            return x
        if self._work is None or self._work.numel() < 3 * n + 64:
            self._work = torch.empty(3 * n + 64, dtype=torch.float64, device="cuda")
        it, fn, cv = C.c_int(), C.c_double(), C.c_int()
        if isinstance(self.op, Matrix):
            plan, kind, opp, vals = self.op.plan, capi.OP_CSR, None, _p(self.op.values)
        else:
            plan, kind, opp, vals = None, capi.OP_PA, self.op.handle, None
        every = 25 if self.check_every is None else self.check_every
        capi.call("femb200_pcg", plan, kind, opp, vals, _p(b), _p(x), n, self.rel_tol, self.abs_tol, self.max_iter,
                  _p(self.dinv), every, int(fixed_iters), _p(self._work), C.byref(it), C.byref(fn),
                  C.byref(cv), _stream())
        self.iterations, self.final_norm, self.converged = it.value, fn.value, bool(cv.value)
        return x


def lifted_rhs(A_nobc_mult, g: np.ndarray, marker: np.ndarray, f: np.ndarray | None = None) -> np.ndarray:
    """b for the linear problem K u = f with u = g on the Dirichlet dofs, in the
    row/column-eliminated form the assembled operator uses (the apply_lifting +
    set_bc sequence of F.cc:822-836 specialised to a linear problem):
    b = f - K_full g on free dofs, b = g on constrained dofs."""
    n = marker.shape[0]
    b = np.zeros(n) if f is None else np.array(f, dtype=np.float64).reshape(n).copy()
    b -= A_nobc_mult(g)
    b[marker != 0] = g[marker != 0]
    return b
