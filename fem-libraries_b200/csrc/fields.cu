// fields.cu -- field operators either side of the hot path (SURVEY.md 8f ranks 3-4).
//
// 1. Damage-field smoothing (M.cc:1258-1315, F.py:160-199): the nodal damage d is spread over the
//    vertex graph of the triangulation by 8 (max_refine + 1) double sweeps
//        s_l = sum over edge neighbours n of d_n      (first sweep: only where d_l < 0.01)
//        d_l = max(s_l / deg_l, d_l)
//    every sweep reading the previous field (Jacobi style: the reference fills a scratch vector
//    first, M.cc:1270-1291).  The Python driver does it with a SciPy adjacency product
//    (F.py:166-186); here it is a gather over the P1 node-block pattern of the plan (the pattern
//    of a P1 triangulation is the edge graph plus the diagonal), one thread per vertex.
// 2. DG0 strain / stress output fields (strainTensor / stressTensor, M.cc:333-430,1551-1563;
//    F.cc:909-942): per cell, the symmetric gradient of u and asym_stress (weight one) at the
//    DG0 node, the cell centroid, stored as (xx, xy, yy).
#include "constitutive.cuh"
#include "element.cuh"
#include "plan.cuh"

namespace femb {

// one sweep: out_l = max(mask_l * sum_n in_n * inv_deg_l, in_l);  MASKED: mask_l = [in_l < thr]
template <bool MASKED>
__global__ void __launch_bounds__(256)
smooth_sweep_kernel(int64_t nv, const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                    const double *__restrict__ din, double *__restrict__ dout, double thr)
{
   const int64_t l = (int64_t)blockIdx.x * 256 + threadIdx.x;
   if (l >= nv) return;
   const double dl = din[l];
   const int64_t b0 = brp[l], b1 = brp[l + 1];
   double s = 0.;
   int deg = 0;
   if (!MASKED || dl < thr)
      for (int64_t k = b0; k < b1; ++k)
      {  // ascending neighbour order, fixed: the result is reproducible bit for bit
         const int32_t n = bcol[k];
         if (n != l) s += din[n], ++deg;
      }
   else
      deg = 1;
   // the reference multiplies by the precomputed reciprocal (M.cc:1247, 1292)
   const double inv = deg > 0 ? 1. / (double)deg : 0.;
   dout[l] = fmax(s * inv, dl);
}

template <int ET>
__global__ void __launch_bounds__(128)
cell_strain_stress_kernel(int64_t ncells, const int32_t *__restrict__ xdofmap, const int32_t *__restrict__ dofmap,
                          const double *__restrict__ x, int xs, const double *__restrict__ E, LameCoef lc,
                          const double *__restrict__ dnod, const double *__restrict__ u, double *__restrict__ strain,
                          double *__restrict__ stress)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv;
   const int64_t e = (int64_t)blockIdx.x * 128 + threadIdx.x;
   if (e >= ncells) return;
   double xv[nv][2], dv[nv];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const int64_t g = xdofmap[e * nv + v];
      xv[v][0] = x[g * xs], xv[v][1] = x[g * xs + 1];
      dv[v] = dnod ? dnod[g] : 0.;
   }
   const double xi = ET == FEMB200_Q2 ? 0.5 : 1. / 3., eta = xi;  // the DG0 node
   double G[nd][2], phi[nv];
   point_geometry<ET>(xv, xi, eta, G, phi);
   double d = 0.;
#pragma unroll
   for (int v = 0; v < nv; ++v) d += phi[v] * dv[v];
   double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;  // grad u (M.cc:343)
#pragma unroll
   for (int a = 0; a < nd; ++a)
   {
      const double2 ua = reinterpret_cast<const double2 *>(u)[dofmap[e * nd + a]];
      g00 += ua.x * G[a][0], g01 += ua.x * G[a][1];
      g10 += ua.y * G[a][0], g11 += ua.y * G[a][1];
   }
   const double sh = 0.5 * (g01 + g10);  // Symmetrize (M.cc:344)
   if (strain) strain[3 * e] = g00, strain[3 * e + 1] = sh, strain[3 * e + 2] = g11;
   if (stress)
   {
      const double eps[4] = {g00, sh, sh, g11};
      double sig[4];
      asym_stress(E[e] * lc.c2, E[e] * lc.c3, d, 1., eps, sig);
      stress[3 * e] = sig[0], stress[3 * e + 1] = sig[1], stress[3 * e + 2] = sig[3];
   }
}

}  // namespace femb

using namespace femb;

extern "C" int femb200_smooth_damage(const femb200_plan *p, double *d_d, double *d_work, int niter, double threshold,
                                     void *stream)
{
   FEMB_CHECK(p && d_d && d_work, "smooth_damage: null argument");
   FEMB_REFUSE_Q1(p->etype, "smooth_damage");
   FEMB_CHECK(p->etype == FEMB200_P1, "smooth_damage: the plan must be the P1 (vertex) plan of the triangulation");
   FEMB_CHECK(niter >= 0, "smooth_damage: negative iteration count");
   cudaStream_t st = as_stream(stream);
   const unsigned grid = (unsigned)cdiv(p->nnodes, 256);
   for (int it = 0; it < niter; ++it)
   {
      smooth_sweep_kernel<true><<<grid, 256, 0, st>>>(p->nnodes, p->brp, p->bcol, d_d, d_work, threshold);
      smooth_sweep_kernel<false><<<grid, 256, 0, st>>>(p->nnodes, p->brp, p->bcol, d_work, d_d, threshold);
   }
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_cell_strain_stress(int etype, int64_t ncells, const int32_t *d_xdofmap, const int32_t *d_dofmap,
                                          const double *d_x, int x_stride, const double *d_E, double nu,
                                          const double *d_dnod, const double *d_u, double *d_strain, double *d_stress,
                                          void *stream)
{
   FEMB_REFUSE_Q1(etype, "cell_strain_stress");
   FEMB_CHECK(etype >= FEMB200_P1 && etype <= FEMB200_Q2, "cell_strain_stress: unknown element family %d", etype);
   FEMB_CHECK(ncells > 0 && d_xdofmap && d_dofmap && d_x && d_u, "cell_strain_stress: null argument");
   FEMB_CHECK(!d_stress || d_E, "cell_strain_stress: the stress needs the Young modulus");
   FEMB_CHECK(x_stride == 2 || x_stride == 3, "cell_strain_stress: x_stride must be 2 or 3, got %d", x_stride);
   cudaStream_t st = as_stream(stream);
   const unsigned grid = (unsigned)cdiv(ncells, 128);
   const LameCoef lc = lame_coef(nu);
   switch (etype)
   {
      case FEMB200_P1:
         cell_strain_stress_kernel<FEMB200_P1><<<grid, 128, 0, st>>>(ncells, d_xdofmap, d_dofmap, d_x, x_stride, d_E, lc,
                                                                      d_dnod, d_u, d_strain, d_stress);
         break;
      case FEMB200_P2:
         cell_strain_stress_kernel<FEMB200_P2><<<grid, 128, 0, st>>>(ncells, d_xdofmap, d_dofmap, d_x, x_stride, d_E, lc,
                                                                      d_dnod, d_u, d_strain, d_stress);
         break;
      default:
         cell_strain_stress_kernel<FEMB200_Q2><<<grid, 128, 0, st>>>(ncells, d_xdofmap, d_dofmap, d_x, x_stride, d_E, lc,
                                                                      d_dnod, d_u, d_strain, d_stress);
   }
   FEMB_LAUNCH_CHECK();
   return 0;
}
