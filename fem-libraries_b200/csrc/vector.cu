// vector.cu -- residual vector assembly and Dirichlet lifting.
//
// Role in the reference: the setF lambda of the FEniCSx driver (F.cc:817-845:
// assemble_vector(F) -> apply_lifting(J, bcs, u, -1) -> ghost update -> set_bc(-1)) and
// ParNonlinearForm::Mult -> damIntegrator::AssembleElementVector + asym_stress on the MFEM
// side (M.cc:559-637, 207-329):
//     r_e = sum_q w_q |det J_q| G_q sigma_q(u)  -  sum_q' w_q' |det J_q'| N(q') f(q')
// stress term with the element's rule (P1: the single point the reference forces), load term
// with the degree-2 3-point rule on triangles (M.cc:613-632) / 3x3 Gauss on quadrilaterals.
//
// B200 design: two passes, both write-once, no atomics, no zero-fill, deterministic.
//   cell_residual_kernel   one thread per cell (coalesced over cells): the whole element vector r_e (2 nd doubles),
//                          stress evaluated once per point of the cell, written to the plan's per-cell scratch through
//                          a shared-memory stage;
//   vector_gather_kernel   one thread per node: walks the cells incident to the node through the plan's visit records
//                          (cell, local index a) and sums the pairs r_e[a] (one 16-byte load each) in list order.
// The single-pass form (assemble_vector_kernel: every visit recomputes its cell's stress and keeps two entries, 12
// evaluations per P2 cell) stays as plan option "vector_path" = 1: 1.60 / 3.06 ms (linear / damaged with load) at n = 1448
// against the two-pass form's cost of a coalesced cell pass + a 16-byte gather per visit.
#include "constitutive.cuh"
#include "element.cuh"
#include "plan.cuh"

namespace femb {

struct VecArgs
{
   int64_t nnodes;
   const int32_t *nptr;
   const VisitRec *vrec;
   const uint8_t *perm;
   const uint16_t *voff;
   const int32_t *xdofmap, *dofmap;
   const double *x;
   int xs;
   const double *E;
   LameCoef lc;
   const double *dnod, *u, *fnod;
   double *b;
};

template <int ET>
__global__ void __launch_bounds__(kAsmR) assemble_vector_kernel(VecArgs A)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq;
   constexpr int LET = (ET == FEMB200_Q2) ? FEMB200_Q2 : FEMB200_P2;  // rule of the load term
   constexpr int lq = Elem<LET>::nq;
   __shared__ int32_t s_voff[kAsmLevels];
   const int rank = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR;
   const int nloc = (int)min((int64_t)kAsmR, A.nnodes - n0);
   if (rank < kAsmLevels) s_voff[rank] = A.voff[(int64_t)blockIdx.x * kAsmLevels + rank];
   __syncthreads();
   if (rank >= nloc) return;
   const int64_t I = n0 + A.perm[n0 + rank];
   const int cnt = A.nptr[I + 1] - A.nptr[I];
   const uint4 *rec = reinterpret_cast<const uint4 *>(A.vrec + A.nptr[n0]) + rank;
   double bx = 0., by = 0.;
   for (int c = 0; c < cnt; ++c)
   {
      const Visit r(rec[s_voff[c]]);
      const int64_t e = r.e;
      const int a = r.a;
      double xv[nv][2], dv[nv];
#pragma unroll
      for (int v = 0; v < nv; ++v)
      {
         const int64_t g = A.xdofmap[e * nv + v];
         xv[v][0] = A.x[g * A.xs], xv[v][1] = A.x[g * A.xs + 1];
         dv[v] = A.dnod ? A.dnod[g] : 0.;
      }
      double ue[nd][2], fe[nd][2];
#pragma unroll
      for (int b = 0; b < nd; ++b)
      {
         const int64_t g = A.dofmap[e * nd + b];
         const double2 uu = reinterpret_cast<const double2 *>(A.u)[g];
         ue[b][0] = uu.x, ue[b][1] = uu.y;
         if (A.fnod)
         {
            const double2 ff = reinterpret_cast<const double2 *>(A.fnod)[g];
            fe[b][0] = ff.x, fe[b][1] = ff.y;
         }
      }
      const double Ee = A.E[e];
      const double lam = Ee * A.lc.c2, mu = Ee * A.lc.c3;
      double rx = 0., ry = 0.;
#pragma unroll 1
      for (int q = 0; q < nq; ++q)
      {
         double G[nd][2], phi[nv];
         const double w = qp_geometry<ET>(xv, q, G, phi);
         double d = 0.;
#pragma unroll
         for (int v = 0; v < nv; ++v) d += phi[v] * dv[v];
         double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;  // grad u (M.cc:742)
         double gax = 0., gay = 0.;
#pragma unroll
         for (int b = 0; b < nd; ++b)
         {
            g00 += ue[b][0] * G[b][0], g01 += ue[b][0] * G[b][1];
            g10 += ue[b][1] * G[b][0], g11 += ue[b][1] * G[b][1];
            if (b == a) gax = G[b][0], gay = G[b][1];
         }
         const double sh = 0.5 * (g01 + g10);
         const double eps[4] = {g00, sh, sh, g11};
         double sig[4];
         asym_stress(lam, mu, d, w, eps, sig);
         rx += gax * sig[0] + gay * sig[2];  // AddMult(gdshape, sig, res), M.cc:601
         ry += gax * sig[1] + gay * sig[3];
      }
      if (A.fnod)
      {
#pragma unroll 1
         for (int q = 0; q < lq; ++q)
         {
            double xi, eta, wq, N[nd], G[nd][2], phi[nv];
            quad_point<LET>(q, xi, eta, wq);
            basis_values<ET>(xi, eta, N);
            // |det J| at the point: qp_geometry returns (its own rule's weight) * |det J|
            double dphi[nv][2];
            geom_basis<ET>(xi, eta, phi, dphi);
            double J00 = 0., J01 = 0., J10 = 0., J11 = 0.;
#pragma unroll
            for (int v = 0; v < nv; ++v)
            {
               J00 += xv[v][0] * dphi[v][0], J01 += xv[v][0] * dphi[v][1];
               J10 += xv[v][1] * dphi[v][0], J11 += xv[v][1] * dphi[v][1];
            }
            const double w = wq * fabs(J00 * J11 - J01 * J10);
            (void)G;
            double f0 = 0., f1 = 0., na = 0.;
#pragma unroll
            for (int b = 0; b < nd; ++b)
            {
               f0 += N[b] * fe[b][0], f1 += N[b] * fe[b][1];
               if (b == a) na = N[b];
            }
            rx -= w * na * f0;  // AddMult_a_VWt(-wl, shape, f, res), M.cc:631
            ry -= w * na * f1;
         }
      }
      bx += rx, by += ry;
   }
   reinterpret_cast<double2 *>(A.b)[I] = make_double2(bx, by);
}

// pass 1 of the two-pass form: r_e of every cell -> cellr[cell][nd][2]
template <int ET>
__global__ void __launch_bounds__(128, ET == FEMB200_Q2 ? 2 : 4) cell_residual_kernel(VecArgs A, int64_t ncells, double *__restrict__ cellr)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq;
   constexpr int LET = (ET == FEMB200_Q2) ? FEMB200_Q2 : FEMB200_P2;  // rule of the load term
   constexpr int lq = Elem<LET>::nq;
   constexpr int RS = 2 * nd, STRIDE = RS + 2;  // 16-byte units of a record: nd; odd stride in units (no bank conflicts)
   __shared__ __align__(16) double stage[4][32 * STRIDE];
   const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
   const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + 32 * warp;
   const int64_t eid = e0 + lane;
   const bool active = eid < ncells;
   const int64_t e = active ? eid : ncells - 1;
   double xv[nv][2], dv[nv];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const int64_t g = A.xdofmap[e * nv + v];
      xv[v][0] = A.x[g * A.xs], xv[v][1] = A.x[g * A.xs + 1];
      dv[v] = A.dnod ? A.dnod[g] : 0.;
   }
   // the nodal loads are gathered after the stress loop (their 2 nd registers would cost a resident CTA: the kernel is
   // bound by the latency of its gathers, i.e. by occupancy)
   double ue[nd][2];
   int32_t gid[nd];
#pragma unroll
   for (int b = 0; b < nd; ++b)
   {
      gid[b] = A.dofmap[e * nd + b];
      const double2 uu = reinterpret_cast<const double2 *>(A.u)[gid[b]];
      ue[b][0] = uu.x, ue[b][1] = uu.y;
   }
   const double Ee = A.E[e];
   const double lam = Ee * A.lc.c2, mu = Ee * A.lc.c3;
   double r[nd][2];
#pragma unroll
   for (int b = 0; b < nd; ++b) r[b][0] = r[b][1] = 0.;
   // triangles: constant Jacobian (one reciprocal per cell)
   double gl[3][2], wtri = 0.;
   if (ET != FEMB200_Q2)
   {
      const double det = (xv[1][0] - xv[0][0]) * (xv[2][1] - xv[0][1]) - (xv[2][0] - xv[0][0]) * (xv[1][1] - xv[0][1]);
      const double id = 1. / det;
      gl[1][0] = (xv[2][1] - xv[0][1]) * id, gl[1][1] = -(xv[2][0] - xv[0][0]) * id;
      gl[2][0] = -(xv[1][1] - xv[0][1]) * id, gl[2][1] = (xv[1][0] - xv[0][0]) * id;
      gl[0][0] = -gl[1][0] - gl[2][0], gl[0][1] = -gl[1][1] - gl[2][1];
      wtri = (ET == FEMB200_P1 ? 0.5 : 1. / 6.) * fabs(det);
   }
#pragma unroll 1
   for (int q = 0; q < nq; ++q)
   {
      double G[nd][2], phi[nv];
      double w;
      if constexpr (ET == FEMB200_Q2)
         w = qp_geometry<ET>(xv, q, G, phi);
      else
      {
         tri_point_grads<ET>(q, gl, G, phi);
         w = wtri;
      }
      double d = 0.;
#pragma unroll
      for (int v = 0; v < nv; ++v) d += phi[v] * dv[v];
      double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;  // grad u (M.cc:742)
#pragma unroll
      for (int b = 0; b < nd; ++b)
      {
         g00 += ue[b][0] * G[b][0], g01 += ue[b][0] * G[b][1];
         g10 += ue[b][1] * G[b][0], g11 += ue[b][1] * G[b][1];
      }
      const double sh = 0.5 * (g01 + g10);
      const double eps[4] = {g00, sh, sh, g11};
      double sig[4];
      asym_stress(lam, mu, d, w, eps, sig);
#pragma unroll
      for (int b = 0; b < nd; ++b)
      {  // AddMult(gdshape, sig, res), M.cc:601
         r[b][0] += G[b][0] * sig[0] + G[b][1] * sig[2];
         r[b][1] += G[b][0] * sig[1] + G[b][1] * sig[3];
      }
   }
   if (A.fnod)
   {
      double fe[nd][2];
#pragma unroll
      for (int b = 0; b < nd; ++b)
      {
         const double2 ff = reinterpret_cast<const double2 *>(A.fnod)[gid[b]];
         fe[b][0] = ff.x, fe[b][1] = ff.y;
      }
#pragma unroll 1
      for (int q = 0; q < lq; ++q)
      {
         double xi, eta, wq, N[nd], phi[nv], dphi[nv][2];
         quad_point<LET>(q, xi, eta, wq);
         basis_values<ET>(xi, eta, N);
         geom_basis<ET>(xi, eta, phi, dphi);
         double J00 = 0., J01 = 0., J10 = 0., J11 = 0.;
#pragma unroll
         for (int v = 0; v < nv; ++v)
         {
            J00 += xv[v][0] * dphi[v][0], J01 += xv[v][0] * dphi[v][1];
            J10 += xv[v][1] * dphi[v][0], J11 += xv[v][1] * dphi[v][1];
         }
         const double w = wq * fabs(J00 * J11 - J01 * J10);
         double f0 = 0., f1 = 0.;
#pragma unroll
         for (int b = 0; b < nd; ++b) f0 += N[b] * fe[b][0], f1 += N[b] * fe[b][1];
#pragma unroll
         for (int b = 0; b < nd; ++b)
         {  // AddMult_a_VWt(-wl, shape, f, res), M.cc:631
            r[b][0] -= w * N[b] * f0;
            r[b][1] -= w * N[b] * f1;
         }
      }
   }
   double2 *R = reinterpret_cast<double2 *>(stage[warp] + lane * STRIDE);
#pragma unroll
   for (int b = 0; b < nd; ++b) R[b] = make_double2(r[b][0], r[b][1]);
   __syncwarp();
   // the 32 records of the warp are one contiguous range of cellr
   const int ncell = (int)max((int64_t)0, min((int64_t)32, ncells - e0));
   for (int t = lane; t < ncell * nd; t += 32)
   {
      const int c = t / nd, k = t - c * nd;
      reinterpret_cast<double2 *>(cellr + e0 * RS)[t] = reinterpret_cast<const double2 *>(stage[warp] + c * STRIDE)[k];
   }
}

// pass 2: b[2I..2I+1] = sum over the visits (cell e, local index a) of node I of r_e[a], in list order
__global__ void __launch_bounds__(kAsmR)
vector_gather_kernel(int64_t nnodes, const int32_t *__restrict__ nptr, const VisitRec *__restrict__ vrec,
                     const uint8_t *__restrict__ perm, const uint16_t *__restrict__ voff, int nd,
                     const double *__restrict__ cellr, double *__restrict__ b)
{
   __shared__ int32_t s_voff[kAsmLevels];
   const int rank = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR;
   const int nloc = (int)min((int64_t)kAsmR, nnodes - n0);
   if (rank < kAsmLevels) s_voff[rank] = voff[(int64_t)blockIdx.x * kAsmLevels + rank];
   __syncthreads();
   if (rank >= nloc) return;
   const int64_t I = n0 + perm[n0 + rank];
   const int cnt = nptr[I + 1] - nptr[I];
   const uint4 *rec = reinterpret_cast<const uint4 *>(vrec + nptr[n0]) + rank;
   const double2 *cr = reinterpret_cast<const double2 *>(cellr);
   double bx = 0., by = 0.;
#pragma unroll 4
   for (int c = 0; c < cnt; ++c)
   {
      const uint4 raw = rec[s_voff[c]];
      const double2 v = cr[(int64_t)raw.x * nd + (raw.y & 0xffu)];
      bx += v.x, by += v.y;
   }
   reinterpret_cast<double2 *>(b)[I] = make_double2(bx, by);
}

// apply_lifting + set_bc on the node rows that have a constrained column (plan list lift_nodes: O(boundary) rows): one warp
// per row, y = sum_J A_IJ w_J with w = (g - u) on the constrained dofs and 0 elsewhere evaluated on the fly, then
// b -= scale * y on the free dofs of the row and b = scale * (g - u) on its constrained ones.  Every other row of
// J[:, bc] (g - u) is exactly zero: b is left alone there.  (Until round 2 this was a full SpMV with a dense w and two
// whole-vector kernels: 13 ms at config 4.)
__global__ void __launch_bounds__(128)
lift_rows_kernel(int nlift, const int32_t *__restrict__ lift_nodes, const uint8_t *__restrict__ bc,
                 const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol, const double *__restrict__ values,
                 const double *__restrict__ g, const double *__restrict__ u, double scale, double *__restrict__ b)
{
   const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
   if (w >= nlift) return;
   const int64_t I = lift_nodes[w], b0 = brp[I];
   const int deg = (int)(brp[I + 1] - b0);
   const double2 *row0 = reinterpret_cast<const double2 *>(values + 4 * b0), *row1 = row0 + deg;
   double y0 = 0., y1 = 0.;
   for (int s = lane; s < deg; s += 32)
   {
      const int64_t J = bcol[b0 + s];
      const double w0 = bc[2 * J] ? g[2 * J] - u[2 * J] : 0., w1 = bc[2 * J + 1] ? g[2 * J + 1] - u[2 * J + 1] : 0.;
      const double2 a = row0[s], c = row1[s];
      y0 += a.x * w0 + a.y * w1;
      y1 += c.x * w0 + c.y * w1;
   }
#pragma unroll
   for (int o = 16; o > 0; o >>= 1)
   {
      y0 += __shfl_xor_sync(0xffffffffu, y0, o);
      y1 += __shfl_xor_sync(0xffffffffu, y1, o);
   }
   if (lane < 2)
   {
      const int64_t i = 2 * I + lane;
      const double y = lane ? y1 : y0;
      b[i] = bc[i] ? scale * (g[i] - u[i]) : b[i] - scale * y;
   }
}

// b = scale * (g - u) on the constrained dofs (dolfinx set_bc, F.cc:836); free dofs untouched
__global__ void set_bc_kernel(int64_t n, const uint8_t *__restrict__ bc, const double *__restrict__ g,
                              const double *__restrict__ u, double scale, double *__restrict__ b)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n && bc[i]) b[i] = scale * (g[i] - u[i]);
}

__global__ void axpy_kernel(int64_t n, double alpha, const double *__restrict__ x, double *__restrict__ y)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n) y[i] += alpha * x[i];
}

}  // namespace femb

using namespace femb;

extern "C" int femb200_set_bc(const femb200_plan *p, const double *d_g, const double *d_u, double scale, double *d_b,
                              void *stream)
{
   FEMB_CHECK(p && d_g && d_u && d_b, "set_bc: null argument");
   FEMB_CHECK(p->bc != nullptr, "set_bc: no Dirichlet dofs set on the plan");
   const int64_t n = 2 * p->nnodes;
   set_bc_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(n, p->bc, d_g, d_u, scale, d_b);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_axpy(int64_t n, double alpha, const double *d_x, double *d_y, void *stream)
{
   FEMB_CHECK(n >= 0 && (n == 0 || (d_x && d_y)), "axpy: bad argument");
   if (n == 0) return 0;
   axpy_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(n, alpha, d_x, d_y);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_assemble_vector(const femb200_plan *p, const double *d_x, int x_stride, const double *d_E,
                                       double nu, const double *d_dnod, const double *d_u, const double *d_fnod,
                                       double *d_b, void *stream)
{
   FEMB_CHECK(p && d_x && d_E && d_u && d_b, "assemble_vector: null argument");
   FEMB_REFUSE_Q1(p->etype, "assemble_vector");
   FEMB_CHECK(x_stride == 2 || x_stride == 3, "assemble_vector: x_stride must be 2 or 3, got %d", x_stride);
   VecArgs A;
   A.nnodes = p->nnodes, A.nptr = p->nptr, A.vrec = p->vrec, A.perm = p->perm, A.voff = p->voff;
   A.xdofmap = p->xdofmap, A.dofmap = p->dofmap, A.x = d_x, A.xs = x_stride, A.E = d_E, A.lc = lame_coef(nu);
   A.dnod = d_dnod, A.u = d_u, A.fnod = d_fnod, A.b = d_b;
   const unsigned grid = (unsigned)cdiv(p->nnodes, kAsmR);
   cudaStream_t st = as_stream(stream);
   if (p->opt_vector_path == 1)
   {  // single pass: every visit recomputes its cell
      switch (p->etype)
      {
         case FEMB200_P1: assemble_vector_kernel<FEMB200_P1><<<grid, kAsmR, 0, st>>>(A); break;
         case FEMB200_P2: assemble_vector_kernel<FEMB200_P2><<<grid, kAsmR, 0, st>>>(A); break;
         default: assemble_vector_kernel<FEMB200_Q2><<<grid, kAsmR, 0, st>>>(A);
      }
      FEMB_LAUNCH_CHECK();
      return 0;
   }
   // two passes through the plan's per-cell scratch (shared with the damage records of the matrix assembly: both are
   // valid inside one call only; one stream per plan at a time)
   femb200_plan *pm = const_cast<femb200_plan *>(p);
   if (int rc = plan_cell_scratch(pm)) return rc;
   const unsigned cgrid = (unsigned)cdiv(p->ncells, 128);
   switch (p->etype)
   {
      case FEMB200_P1: cell_residual_kernel<FEMB200_P1><<<cgrid, 128, 0, st>>>(A, p->ncells, pm->celld); break;
      case FEMB200_P2: cell_residual_kernel<FEMB200_P2><<<cgrid, 128, 0, st>>>(A, p->ncells, pm->celld); break;
      default: cell_residual_kernel<FEMB200_Q2><<<cgrid, 128, 0, st>>>(A, p->ncells, pm->celld);
   }
   FEMB_LAUNCH_CHECK();
   vector_gather_kernel<<<grid, kAsmR, 0, st>>>(p->nnodes, p->nptr, p->vrec, p->perm, p->voff, p->nd, pm->celld, d_b);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_apply_lifting(const femb200_plan *p, const double *d_values_nobc, const double *d_g,
                                     const double *d_u, double scale, double *d_b, double *d_work, void *stream)
{
   FEMB_CHECK(p && d_values_nobc && d_g && d_u && d_b, "apply_lifting: null argument");
   FEMB_REFUSE_Q1(p->etype, "apply_lifting");
   FEMB_CHECK(p->bc != nullptr, "apply_lifting: no Dirichlet dofs set on the plan");
   (void)d_work;  // scratch of the former SpMV form; kept in the signature
   if (p->nlift == 0) return 0;
   lift_rows_kernel<<<(unsigned)cdiv((int64_t)p->nlift * 32, 128), 128, 0, as_stream(stream)>>>(
       p->nlift, p->lift_nodes, p->bc, p->brp, p->bcol, d_values_nobc, d_g, d_u, scale, d_b);
   FEMB_LAUNCH_CHECK();
   return 0;
}
