// element.cu -- batched element tangent kernel.
//
// Drop-in for the per-cell ufcx `tabulate_tensor` of form J (manual.py:102) and
// for damIntegrator::AssembleElementGrad (M.cc:639-916): one launch tabulates
// every cell.  K_e = sum_q w_q |det J_q| B_q D_q B_q^t  (SURVEY.md A.1, A.9).
#include "constitutive.cuh"
#include "element.cuh"

namespace femb {

// Block (a, b) of the element matrix of an undamaged straight-sided triangle from the nine P1 blocks
// W[c][d] = |T| B_c D B_d^t (c, d = vertices; M.cc:699-704, 885-887 with w = |T|): what the 3-point rule integrates
// exactly (SURVEY.md A.9; derivation in assemble.cu), at ~0.6 kflop per P2 element instead of 4.3 kflop for the
// triple product per point:
//   vertex / vertex          W^{aa}, or -W^{ab} / 3
//   vertex a / edge (r, s)   4/3 W^{as} if a = r, 4/3 W^{ar} if a = s, 0 if a is opposite; edge / vertex likewise
//   edge (p, q) / edge (r, s)  4/3 [(1 + d_qs) W^{pr} + (1 + d_qr) W^{ps} + (1 + d_ps) W^{qr} + (1 + d_pr) W^{qs}]
// a, b are compile-time constants at every call site (unrolled loops): W stays in registers.
template <int ET>
__device__ __forceinline__ void closed_block(int a, int b, const double (*W)[3][4], double *k)
{
   if (ET == FEMB200_P1)
   {
#pragma unroll
      for (int j = 0; j < 4; ++j) k[j] = W[a][b][j];
      return;
   }
   const double c43 = 4. / 3.;
   // edge 3 + i joins the two vertices other than i
   const int p = (a - 3 + 1) % 3, q = (a - 3 + 2) % 3, r = (b - 3 + 1) % 3, t = (b - 3 + 2) % 3;
   if (a < 3 && b < 3)
   {
      const double c = a == b ? 1. : -1. / 3.;
#pragma unroll
      for (int j = 0; j < 4; ++j) k[j] = c * W[a][b][j];
   }
   else if (a < 3)
   {
      const int o = a == r ? t : r;  // the other end of the edge, when a is one of its ends
#pragma unroll
      for (int j = 0; j < 4; ++j) k[j] = (a == r || a == t) ? c43 * W[a][o][j] : 0.;
   }
   else if (b < 3)
   {
      const int o = b == p ? q : p;
#pragma unroll
      for (int j = 0; j < 4; ++j) k[j] = (b == p || b == q) ? c43 * W[o][b][j] : 0.;
   }
   else
   {
      const double cpr = q == t ? 2. : 1., cps = q == r ? 2. : 1., cqr = p == t ? 2. : 1., cqs = p == r ? 2. : 1.;
#pragma unroll
      for (int j = 0; j < 4; ++j)
         k[j] = c43 * (cpr * W[p][r][j] + cps * W[p][t][j] + cqr * W[q][r][j] + cqs * W[q][t][j]);
   }
}

// One thread integrates one cell; the 2 x n slabs of the element matrix (a row pair in the ufcx layout, a column
// pair in the MFEM layout) go through a per-warp shared-memory stage (padded: conflict-free 16-byte accesses) and
// leave as contiguous n-double chunks, 12 lanes per 96-byte chunk for P2: every 32-byte sector written whole,
// instead of 32 lanes storing 1152 bytes apart (5.1 -> 1.46 ms for 4.19 M P2 cells; with the closed form of the undamaged
// cells 0.84 ms = 0.92 of the HBM roofline; compiled for 4 CTAs per SM, 128 registers: 0.87 ms, not kept).
template <int ET, bool ROWMAJOR>
__global__ void __launch_bounds__(128)
tabulate_kernel(int64_t ncells, double *__restrict__ A, const double *__restrict__ x, int xs,
                const int32_t *__restrict__ xdofmap, const int32_t *__restrict__ dofmap, const double *__restrict__ E,
                LameCoef lc, const double *__restrict__ dnod, const double *__restrict__ u, int variant)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq, n = 2 * nd;
   // P1: the whole 6 x 6 matrix of a cell is staged, the 32 matrices of a warp leave as one contiguous 9 KB range;
   // P2 / Q2: one slab (2 x n) at a time
   constexpr bool FULL = ET == FEMB200_P1;
   constexpr int STRIDE = FULL ? n * n + 2 : 2 * n + 2;  // doubles per lane in the stage
   __shared__ __align__(16) double stage[4][32 * STRIDE];
   const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   const bool active = e < ncells;
   const int64_t ec = active ? e : ncells - 1;  // idle lanes of the last warp repeat the last cell, store nothing
   const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + 32 * warp;  // first cell of this warp
   const int nwarp = (int)max((int64_t)0, min((int64_t)32, ncells - e0));

   double xv[nv][2], dv[nv];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const int64_t g = xdofmap[ec * nv + v];
      xv[v][0] = x[g * xs];
      xv[v][1] = x[g * xs + 1];
      dv[v] = dnod ? dnod[g] : 0.;
   }
   const double Ee = E[ec];
   const double lam = Ee * lc.c2, mu = Ee * lc.c3;  // M.cc:1093-1098

   // undamaged straight-sided triangle: closed form from the nine P1 blocks (the cells of a linear problem, and the
   // undamaged cells of a damaged one); everything else integrates point by point
   bool lin = false;
   double W[3][3][4];
   if (ET != FEMB200_Q2)
   {
      lin = true;
#pragma unroll
      for (int q = 0; q < nq; ++q)
      {
         double dN[nd][2], phi[3], w2;
         double xi, eta, wq;
         quad_point<ET>(q, xi, eta, wq);
         (void)dN, (void)w2, (void)wq;
         phi[0] = 1. - xi - eta, phi[1] = xi, phi[2] = eta;
         lin = lin && !(phi[0] * dv[0] + phi[1] * dv[1] + phi[2] * dv[2] > 0.);
      }
      if (lin)
      {
         const double det = (xv[1][0] - xv[0][0]) * (xv[2][1] - xv[0][1]) - (xv[2][0] - xv[0][0]) * (xv[1][1] - xv[0][1]);
         const double id = 1. / det;
         double gl[3][2], Dh[9];
         gl[1][0] = (xv[2][1] - xv[0][1]) * id, gl[1][1] = -(xv[2][0] - xv[0][0]) * id;
         gl[2][0] = -(xv[1][1] - xv[0][1]) * id, gl[2][1] = (xv[1][0] - xv[0][0]) * id;
         gl[0][0] = -gl[1][0] - gl[2][0], gl[0][1] = -gl[1][1] - gl[2][1];
         hooke_scaled(lam, mu, 1., Dh);
         const double wT = 0.5 * fabs(det);
#pragma unroll
         for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d)
            {
               W[c][d][0] = W[c][d][1] = W[c][d][2] = W[c][d][3] = 0.;
               bdb_block(gl[c], gl[d], Dh, wT, W[c][d]);
            }
      }
   }
   constexpr bool rowmajor = ROWMAJOR;
   double *st = stage[warp] + lane * STRIDE;
   auto put = [&](int a, int b, const double *k) {
      if (rowmajor)
      {  // chunk r = row 2a + r: entries (2b, 2b + 1)
         double *s0 = FULL ? st + 2 * a * n : st;
         reinterpret_cast<double2 *>(s0)[b] = make_double2(k[0], k[1]);
         reinterpret_cast<double2 *>(s0 + n)[b] = make_double2(k[2], k[3]);
      }
      else
      {  // chunk c = column c * nd + b: rows a and nd + a (elmat(i, j) at i + j n, M.cc:647,673)
         double *s0 = FULL ? st + b * n : st, *s1 = FULL ? st + (nd + b) * n : st + n;
         s0[a] = k[0], s0[nd + a] = k[2];
         s1[a] = k[1], s1[nd + a] = k[3];
      }
   };
   auto flush = [&](const int o) {  // slab o of the warp's cells leaves: 2 chunks of n doubles per cell, n double2 units per cell
      if (FULL)
      {
         if (o != nd - 1) return;
         __syncwarp();
         constexpr int UPC = n * n / 2;  // 16-byte units per cell
         double2 *dst = reinterpret_cast<double2 *>(A + e0 * (int64_t)(n * n));
         for (int t = lane; t < nwarp * UPC; t += 32)
         {
            const int c = t / UPC, r = t - c * UPC;
            dst[t] = reinterpret_cast<const double2 *>(stage[warp] + c * STRIDE)[r];
         }
         return;
      }
      __syncwarp();
      for (int t = lane; t < nwarp * n; t += 32)
      {
         const int c = t / n, r = t - c * n;       // cell of the warp, unit in its slab
         const int ch = r / nd, j = r - ch * nd;   // chunk, double2 inside the chunk
         const double2 val = reinterpret_cast<const double2 *>(stage[warp] + c * STRIDE + ch * n)[j];
         double *dst = A + (e0 + c) * (int64_t)(n * n) + (rowmajor ? (int64_t)(2 * o + ch) * n : (int64_t)(ch * nd + o) * n);
         reinterpret_cast<double2 *>(dst)[j] = val;
      }
      __syncwarp();
   };
   // slab o: rows (2o, 2o+1) of the ufcx layout / columns (o, nd + o) of the MFEM layout.  A warp whose 32 cells are all
   // undamaged triangles takes the closed form with the slab loop unrolled (closed_block needs constant node numbers);
   // any other warp integrates all its cells point by point with rolled loops (G indexed in local memory, L1 hits).
   if (ET != FEMB200_Q2 && __all_sync(0xffffffffu, lin))
   {
#pragma unroll
      for (int o = 0; o < nd; ++o)
      {
#pragma unroll
         for (int i = 0; i < nd; ++i)
         {
            const int a = rowmajor ? o : i, b = rowmajor ? i : o;
            double k[4];
            closed_block<ET>(a, b, W, k);
            put(a, b, k);
         }
         flush(o);
      }
      return;
   }
   double G[nq][nd][2], w[nq], D[nq][9];
   if constexpr (ET == FEMB200_Q2)
   {
#pragma unroll
      for (int q = 0; q < nq; ++q)
      {
         double phi[nv];
         w[q] = qp_geometry<ET>(xv, q, G[q], phi);
         double d = 0.;
#pragma unroll
         for (int v = 0; v < nv; ++v) d += phi[v] * dv[v];
         if (d > 0.)
         {
            double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;  // grad u (M.cc:742)
            if (u)
#pragma unroll
               for (int a = 0; a < nd; ++a)
               {
                  const int64_t gd = 2 * (int64_t)dofmap[ec * nd + a];
                  const double ux = u[gd], uy = u[gd + 1];
                  g00 += ux * G[q][a][0];
                  g01 += ux * G[q][a][1];
                  g10 += uy * G[q][a][0];
                  g11 += uy * G[q][a][1];
               }
            const double s = 0.5 * (g01 + g10);
            const double eps[4] = {g00, s, s, g11};
            tangent(variant, lam, mu, d, eps, D[q]);
         }
         else
            hooke_scaled(lam, mu, 1., D[q]);
      }
   }
   else
   {  // triangles: u gathered once per cell, before the points
      bool dam = false;  // d > 0 at some point of the cell: the tangent needs grad u
      double dq[nq];
#pragma unroll
      for (int q = 0; q < nq; ++q)
      {
         double phi[nv];
         w[q] = qp_geometry<ET>(xv, q, G[q], phi);
         dq[q] = 0.;
#pragma unroll
         for (int v = 0; v < nv; ++v) dq[q] += phi[v] * dv[v];
         dam = dam || dq[q] > 0.;
      }
      double ue[nd][2];
      if (dam)
      {
#pragma unroll
         for (int a = 0; a < nd; ++a)
         {
            const int64_t gd = 2 * (int64_t)dofmap[ec * nd + a];
            ue[a][0] = u ? u[gd] : 0., ue[a][1] = u ? u[gd + 1] : 0.;
         }
      }
#pragma unroll 1
      for (int q = 0; q < nq; ++q)
      {
         if (dq[q] > 0.)
         {
            double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;  // grad u (M.cc:742)
#pragma unroll
            for (int a = 0; a < nd; ++a)
            {
               g00 += ue[a][0] * G[q][a][0];
               g01 += ue[a][0] * G[q][a][1];
               g10 += ue[a][1] * G[q][a][0];
               g11 += ue[a][1] * G[q][a][1];
            }
            const double s = 0.5 * (g01 + g10);
            const double eps[4] = {g00, s, s, g11};
            tangent(variant, lam, mu, dq[q], eps, D[q]);
         }
         else
            hooke_scaled(lam, mu, 1., D[q]);
      }
   }
#pragma unroll 1
   for (int o = 0; o < nd; ++o)
   {
#pragma unroll 1
      for (int i = 0; i < nd; ++i)
      {
         const int a = rowmajor ? o : i, b = rowmajor ? i : o;
         double k[4] = {0., 0., 0., 0.};
#pragma unroll
         for (int q = 0; q < nq; ++q) bdb_block(G[q][a], G[q][b], D[q], w[q], k);
         put(a, b, k);
      }
      flush(o);
   }
}

}  // namespace femb

using namespace femb;

extern "C" int femb200_tabulate_tensor_batched(int etype, int64_t ncells, double *d_A, const double *d_x, int x_stride,
                                               const int32_t *d_xdofmap, const int32_t *d_dofmap, const double *d_E,
                                               double nu, const double *d_dnod, const double *d_u, int variant,
                                               int layout, void *stream)
{
   FEMB_REFUSE_Q1(etype, "tabulate");
   FEMB_CHECK(etype >= FEMB200_P1 && etype <= FEMB200_Q2, "tabulate: unknown element family %d", etype);
   FEMB_CHECK(x_stride == 2 || x_stride == 3, "tabulate: x_stride must be 2 or 3, got %d", x_stride);
   FEMB_CHECK(d_A && d_x && d_xdofmap && d_dofmap && d_E, "tabulate: null pointer argument");
   FEMB_CHECK((reinterpret_cast<uintptr_t>(d_A) & 15) == 0, "tabulate: d_A must be 16-byte aligned");
   FEMB_CHECK(layout == FEMB200_ROWMAJOR_INTERLEAVED || layout == FEMB200_COLMAJOR_BYNODES, "tabulate: bad layout %d",
              layout);
   if (ncells <= 0) return 0;
   const LameCoef lc = lame_coef(nu);
   const unsigned grid = (unsigned)cdiv(ncells, 128);
   cudaStream_t st = as_stream(stream);
   const bool rm = layout == FEMB200_ROWMAJOR_INTERLEAVED;
#define FEMB_TAB(ET)                                                                                                     \
   if (rm)                                                                                                               \
      tabulate_kernel<ET, true><<<grid, 128, 0, st>>>(ncells, d_A, d_x, x_stride, d_xdofmap, d_dofmap, d_E, lc, d_dnod,  \
                                                      d_u, variant);                                                     \
   else                                                                                                                  \
      tabulate_kernel<ET, false><<<grid, 128, 0, st>>>(ncells, d_A, d_x, x_stride, d_xdofmap, d_dofmap, d_E, lc, d_dnod, \
                                                       d_u, variant)
   switch (etype)
   {
      case FEMB200_P1: FEMB_TAB(FEMB200_P1); break;
      case FEMB200_P2: FEMB_TAB(FEMB200_P2); break;
      default: FEMB_TAB(FEMB200_Q2);
   }
#undef FEMB_TAB
   FEMB_LAUNCH_CHECK();
   return 0;
}

// ---- the ufcx kernel signature -----------------------------------------------------------------
// `ufcx_tabulate_tensor_float64` (ufcx.h of ffcx 0.8, un-vendored; corroborated by the generated-kernel patch
// FEniCSx/mechanic2d/addprofile:6-9 and by the form look-ups F.cc:31-67): what a dolfinx Form holds as its cell
// kernel for the bilinear form J of manual.py:102 and calls once per cell.  Batch of one with the device staging
// inside: A (6 x 6 row-major, interleaved dofs, caller-owned, pre-zeroed by the caller) is ACCUMULATED into, as
// ffcx kernels do; no return value (ufcx has no error channel: on a CUDA failure A is left untouched and the
// message is in femb200_last_error()).  Coefficient packing as the form file creates them (manual.py:19,22,30):
//   w = [d0, d1, d2,  E,  u0x, u0y, u1x, u1y, u2x, u2y],  c = [nu],  coordinate_dofs = 3 x (x, y, z).
// Re-entrant: the device scratch is per host thread.  This is the parity surface of the FEniCSx side; the fast path
// is femb200_tabulate_tensor_batched / femb200_assemble_matrix.
namespace femb {
struct UfcxScratch
{
   double *d = nullptr;   // x[9] | E[1] | dnod[3] | u[6] | pad | A[36] (16-byte aligned)
   int32_t *map = nullptr;
};
static UfcxScratch *ufcx_scratch()
{
   static thread_local UfcxScratch s;
   if (!s.d)
   {
      const int32_t id[3] = {0, 1, 2};
      if (cudaMalloc(&s.d, sizeof(double) * 56) != cudaSuccess || cudaMalloc(&s.map, sizeof(id)) != cudaSuccess ||
          cudaMemcpy(s.map, id, sizeof(id), cudaMemcpyHostToDevice) != cudaSuccess)
      {
         set_error("tabulate_tensor_ufcx: device scratch: %s", cudaGetErrorString(cudaGetLastError()));
         cudaFree(s.d), cudaFree(s.map);
         s.d = nullptr, s.map = nullptr;
         return nullptr;
      }
   }
   return &s;
}
}  // namespace femb

extern "C" void femb200_tabulate_tensor_ufcx(double *A, const double *w, const double *c, const double *coordinate_dofs,
                                             const int *entity_local_index, const uint8_t *quadrature_permutation)
{
   (void)entity_local_index, (void)quadrature_permutation;  // cell integrals use neither
   if (!A || !w || !c || !coordinate_dofs)
   {
      set_error("tabulate_tensor_ufcx: null argument");
      return;
   }
   UfcxScratch *s = ufcx_scratch();
   if (!s) return;
   double h[19];
   for (int i = 0; i < 9; ++i) h[i] = coordinate_dofs[i];
   h[9] = w[3];
   for (int i = 0; i < 3; ++i) h[10 + i] = w[i];
   for (int i = 0; i < 6; ++i) h[13 + i] = w[4 + i];
   const bool damaged = w[0] != 0. || w[1] != 0. || w[2] != 0.;
   if (cudaMemcpy(s->d, h, sizeof(h), cudaMemcpyHostToDevice) != cudaSuccess)
   {
      set_error("tabulate_tensor_ufcx: H2D: %s", cudaGetErrorString(cudaGetLastError()));
      return;
   }
   if (femb200_tabulate_tensor_batched(FEMB200_P1, 1, s->d + 20, s->d, 3, s->map, s->map, s->d + 9, c[0],
                                       damaged ? s->d + 10 : nullptr, s->d + 13, FEMB200_TANGENT_CLOSED,
                                       FEMB200_ROWMAJOR_INTERLEAVED, nullptr))
      return;
   double out[36];
   if (cudaMemcpy(out, s->d + 20, sizeof(out), cudaMemcpyDeviceToHost) != cudaSuccess)
   {
      set_error("tabulate_tensor_ufcx: D2H: %s", cudaGetErrorString(cudaGetLastError()));
      return;
   }
   for (int i = 0; i < 36; ++i) A[i] += out[i];
}
