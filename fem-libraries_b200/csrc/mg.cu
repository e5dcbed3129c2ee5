// mg.cu -- geometric multigrid preconditioner on a nested mesh hierarchy.
//
// Levels 0 (the operator being solved, Dirichlet rows / columns applied: an assembled CSR plan, or a matrix-free P2 / Q2
// operator) .. L (coarsest).  Level l + 1 is a P1 or Q1 space on a mesh whose nodes the fine nodes of level l refer to
// through one transfer map of width 2 or 4 (femb200.h): per fine node the coarse node ids of its coincident node, its
// coarse edge (a, b) or its coarse quad; each distinct entry weighs 1 / (number of distinct entries).  The same weights
// act on both components of a node.  P has zero rows for the constrained fine dofs and zero columns for the constrained
// coarse dofs (the per-dof markers of the levels).  A matrix-free level 0 gets its first coarse operator from the
// element Galerkin step of pa.cu (a p-coarsening: sum over the cells of P_e^T K_e P_e), without a fine matrix.
//
//   Galerkin      A_{l+1} = P^T A_l P, gather form: one group of lanes per coarse node row, one lane per 2x2 output
//                 block, accumulated in registers and written once; the pattern is the coarse mesh's own P1 / Q1
//                 pattern (every fine pair (i, j) lies in one coarse cell and every non-zero of P for i or j is a vertex
//                 of that cell), then the coarse Dirichlet rows / columns get a unit diagonal (femb200_apply_dirichlet).
//                 The fine rows a coarse row reads -- its coincident node and one midpoint or quad centre per
//                 off-diagonal block -- are resolved once at create time into `slot_fine` (aligned with the coarse bcol).
//   smoother      Chebyshev of degree k on D^-1 A over [lo lambda, lambda], lambda = 1.1 x a 15-step power iteration
//                 from a fixed seed; the same polynomial before and after the coarse correction (symmetric V(k,k)).
//                 A d goes through femb200_spmv (the matrix-free apply on a matrix-free level 0); the recurrence
//                 r -= D^-1 A d, d = c1 d + c2 r, x += d is one pass.
//   transfers     r_c = P^T (b - A x) in gather form (one thread per coarse node), x += P x_c (one per fine node).
//   coarsest      x = C b with C the dense inverse handed in by the caller (femb200_mg_set_coarse_inverse).
//   PCG           mfem::CGSolver semantics with B = one V-cycle (nom = <B r, r>), the scalar kernels of cg.cu.
// Deterministic: no atomics on values, every sum in a fixed order.
#include <math.h>

#include <algorithm>
#include <vector>

#include "cg_slots.cuh"
#include "plan.cuh"
#include "reduce.cuh"

namespace femb {

namespace {

constexpr int kMgThreads = 256;
constexpr int kMaxDegree = 16;  // Chebyshev degree
constexpr int kPowerIters = 15;
constexpr uint64_t kPowerSeed = 0x6d67706f77657231ull;


struct MgLevel
{
   femb200_plan *plan = nullptr;     // borrowed; level 0: the fine plan, or null for a matrix-free level 0
   const femb200_pa *pa = nullptr;   // borrowed; level 0 of a matrix-free operator
   int64_t nnodes = 0, n = 0;
   const double *values = nullptr;  // level 0: borrowed from setup (null when matrix-free); else = own_values
   double *own_values = nullptr;    // [nnz]
   double *dinv = nullptr, *r = nullptr, *d = nullptr, *t = nullptr;  // [n]
   double *b = nullptr, *x = nullptr;                                   // [n], levels >= 1
   double lambda = 0.;
   double inv_theta = 0., c1[kMaxDegree] = {}, c2[kMaxDegree] = {};
   // transfer to level + 1
   int32_t *map = nullptr;        // [nnodes][width]
   int32_t *slot_fine = nullptr;  // [nnzb of level + 1]
   int group = 0;                 // lanes per coarse row of the Galerkin kernel (level + 1 rows)
};

__device__ __forceinline__ double hash_uniform(uint64_t i)
{
   uint64_t z = kPowerSeed + (i + 1) * 0x9e3779b97f4a7c15ull;
   z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
   z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
   z ^= z >> 31;
   return (double)(z >> 11) * 0x1.0p-52 - 1.;  // [-1, 1)
}

__device__ __forceinline__ int find_col(const int32_t *__restrict__ bcol, int64_t b0, int nb, int col)
{
   for (int k = 0; k < nb; ++k)
      if (bcol[b0 + k] == col) return k;
   return -1;
}

// One row of a transfer map of width W (2 or 4): the coarse node ids of a fine node.
template <int W>
struct MapRow
{
   int m[W];
};

template <int W>
__device__ __forceinline__ MapRow<W> load_map(const int32_t *__restrict__ map, int64_t i)
{
   MapRow<W> r;
   if constexpr (W == 2)
   {
      const int2 v = reinterpret_cast<const int2 *>(map)[i];
      r.m[0] = v.x, r.m[1] = v.y;
   }
   else
   {
      const int4 v = reinterpret_cast<const int4 *>(map)[i];
      r.m[0] = v.x, r.m[1] = v.y, r.m[2] = v.z, r.m[3] = v.w;
   }
   return r;
}

// weight of coarse node J in the interpolation of the fine node: 1 / (number of distinct entries) when J is one of them.
// Pairs: 1 for a coincident node, 1/2 for a midpoint.  Width 4 (rows validated by mg_slots_kernel): (a, a, a, a) 1,
// (a, b, a, b) 1/2, a quad centre 1/4.
template <int W>
__device__ __forceinline__ double map_weight(const MapRow<W> &r, int J)
{
   if constexpr (W == 2)
      return 0.5 * ((r.m[0] == J) + (r.m[1] == J));
   else
   {
      if (r.m[0] != J && r.m[1] != J && r.m[2] != J && r.m[3] != J) return 0.;
      return r.m[0] == r.m[3] ? 1. : (r.m[0] == r.m[2] ? 0.5 : 0.25);
   }
}

// slot_fine[s] = the fine node whose coarse pairs include the block slot s of the coarse pattern: entry k of its map row
// and its partner W - 1 - k name the slot (map[k], map[W-1-k]): the diagonal block of a coincident node, the two blocks
// of the edge of a midpoint, the four blocks of the two diagonals of a quad centre.  err: 1 map entry out of range,
// 2 a pair that is not in the coarse pattern, 3 two fine nodes on one coarse slot, 4 a coarse slot without one,
// 5 a width-4 row that is none of (a, a, a, a), (a, b, a, b), four distinct nodes.
template <int W>
__global__ void mg_slots_kernel(int64_t nf, const int32_t *__restrict__ map, int64_t nc, const int64_t *__restrict__ cbrp,
                                const int32_t *__restrict__ cbcol, int32_t *__restrict__ slot_fine, int *__restrict__ err)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= nf) return;
   const MapRow<W> r = load_map<W>(map, i);
#pragma unroll
   for (int k = 0; k < W; ++k)
      if (r.m[k] < 0 || r.m[k] >= nc)
      {
         *err = 1;
         return;
      }
   if constexpr (W == 4)
   {
      const int *m = r.m;
      const bool co = m[0] == m[1] && m[1] == m[2] && m[2] == m[3];
      const bool edge = m[0] == m[2] && m[1] == m[3] && m[0] != m[1];
      const bool quad = m[0] != m[1] && m[0] != m[2] && m[0] != m[3] && m[1] != m[2] && m[1] != m[3] && m[2] != m[3];
      if (!co && !edge && !quad)
      {
         *err = 5;
         return;
      }
   }
#pragma unroll
   for (int k = 0; k < W; ++k)
   {
      const int a = r.m[k], b = r.m[W - 1 - k];
      const int64_t ba = cbrp[a];
      const int ka = find_col(cbcol, ba, (int)(cbrp[a + 1] - ba), b);
      if (ka < 0)
      {
         *err = 2;
         return;
      }
      slot_fine[ba + ka] = (int32_t)i;
   }
}

template <int W>
__global__ void mg_slots_check_kernel(int64_t nf, const int32_t *__restrict__ map, const int64_t *__restrict__ cbrp,
                                      const int32_t *__restrict__ cbcol, const int32_t *__restrict__ slot_fine,
                                      int64_t nnzb_c, int *__restrict__ err)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < nnzb_c && slot_fine[i] < 0) *err = 4;
   if (i >= nf || *err == 1 || *err == 2 || *err == 5) return;
   const MapRow<W> r = load_map<W>(map, i);
#pragma unroll
   for (int k = 0; k < W; ++k)
   {
      const int64_t ba = cbrp[r.m[k]];
      const int ka = find_col(cbcol, ba, (int)(cbrp[r.m[k] + 1] - ba), r.m[W - 1 - k]);
      if (slot_fine[ba + ka] != (int32_t)i) *err = 3;
   }
}

// A_c = P^T A P.  G lanes per coarse node row I (G >= its block degree); lane k owns the output block (I, J = bcol[k])
// and scans the fine rows of the row (slot_fine) and their fine blocks in a fixed order, accumulating the fine blocks
// (i, j) whose column node j has a weight on J.  Values layout (femb200.h): A[2i + ci, 2j + cj] at
// 4 brp[i] + 2 ci deg(i) + 2 (slot of j) + cj.
template <int G, int W>
__global__ void __launch_bounds__(kMgThreads)
mg_rap_kernel(int64_t nc, const int64_t *__restrict__ cbrp, const int32_t *__restrict__ cbcol,
              const int32_t *__restrict__ slot_fine, const int64_t *__restrict__ fbrp, const int32_t *__restrict__ fbcol,
              const double *__restrict__ fval, const int32_t *__restrict__ map, const uint8_t *__restrict__ fbc,
              double *__restrict__ cval)
{
   const int64_t I = ((int64_t)blockIdx.x * kMgThreads + threadIdx.x) / G;
   const int k = threadIdx.x % G;
   if (I >= nc) return;
   const int64_t cb = cbrp[I];
   const int nb = (int)(cbrp[I + 1] - cb);
   const int J = k < nb ? cbcol[cb + k] : -1;
   double a00 = 0., a01 = 0., a10 = 0., a11 = 0.;
   for (int p = 0; p < nb; ++p)
   {
      const int64_t i = slot_fine[cb + p];
      const double wi = map_weight<W>(load_map<W>(map, i), (int)I);
      const double wi0 = (fbc && fbc[2 * i]) ? 0. : wi, wi1 = (fbc && fbc[2 * i + 1]) ? 0. : wi;
      const int64_t fb = fbrp[i];
      const int fdeg = (int)(fbrp[i + 1] - fb);
      const double *row0 = fval + 4 * fb, *row1 = row0 + 2 * fdeg;
      for (int q = 0; q < fdeg; ++q)
      {
         const int64_t j = fbcol[fb + q];
         const double wj = map_weight<W>(load_map<W>(map, j), J);
         if (wj == 0.) continue;
         const double wj0 = (fbc && fbc[2 * j]) ? 0. : wj, wj1 = (fbc && fbc[2 * j + 1]) ? 0. : wj;
         const double2 v0 = *reinterpret_cast<const double2 *>(row0 + 2 * q);
         const double2 v1 = *reinterpret_cast<const double2 *>(row1 + 2 * q);
         a00 = __fma_rn(__dmul_rn(wi0, wj0), v0.x, a00);
         a01 = __fma_rn(__dmul_rn(wi0, wj1), v0.y, a01);
         a10 = __fma_rn(__dmul_rn(wi1, wj0), v1.x, a10);
         a11 = __fma_rn(__dmul_rn(wi1, wj1), v1.y, a11);
      }
   }
   if (k < nb)
   {
      *reinterpret_cast<double2 *>(cval + 4 * cb + 2 * k) = make_double2(a00, a01);
      *reinterpret_cast<double2 *>(cval + 4 * cb + 2 * nb + 2 * k) = make_double2(a10, a11);
   }
}

// bc[2I + c] = (P^T (b - t))[2I + c], one thread per coarse node; t = A x or null (x = 0)
template <int W>
__global__ void __launch_bounds__(kMgThreads)
mg_restrict_kernel(int64_t nc, const int64_t *__restrict__ cbrp, const int32_t *__restrict__ slot_fine,
                   const int32_t *__restrict__ map, const uint8_t *__restrict__ fbc, const uint8_t *__restrict__ cbc,
                   const double2 *__restrict__ b, const double2 *__restrict__ t, double2 *__restrict__ out)
{
   const int64_t I = (int64_t)blockIdx.x * kMgThreads + threadIdx.x;
   if (I >= nc) return;
   const int64_t cb = cbrp[I];
   const int nb = (int)(cbrp[I + 1] - cb);
   double s0 = 0., s1 = 0.;
   for (int p = 0; p < nb; ++p)
   {
      const int64_t i = slot_fine[cb + p];
      const double w = map_weight<W>(load_map<W>(map, i), (int)I);
      const double w0 = (fbc && fbc[2 * i]) ? 0. : w, w1 = (fbc && fbc[2 * i + 1]) ? 0. : w;
      const double2 bi = b[i];
      const double2 ti = t ? t[i] : make_double2(0., 0.);
      s0 = __fma_rn(w0, __dsub_rn(bi.x, ti.x), s0);
      s1 = __fma_rn(w1, __dsub_rn(bi.y, ti.y), s1);
   }
   if (cbc)
   {
      if (cbc[2 * I]) s0 = 0.;
      if (cbc[2 * I + 1]) s1 = 0.;
   }
   out[I] = make_double2(s0, s1);
}

// x += P x_c, one thread per fine node: (P x_c)_i summed over the distinct coarse nodes in ascending id, as a CSR
// product with sorted columns does (the weights 1, 1/2, 1/4 make every product exact)
template <int W>
__global__ void __launch_bounds__(kMgThreads)
mg_prolong_kernel(int64_t nf, const int32_t *__restrict__ map, const uint8_t *__restrict__ fbc,
                  const uint8_t *__restrict__ cbc, const double *__restrict__ xc, double *__restrict__ x)
{
   const int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x;
   if (i >= nf) return;
   const MapRow<W> r = load_map<W>(map, i);
   int cn[W], nd = 0;  // distinct entries, ascending
#pragma unroll
   for (int k = 0; k < W; ++k)
   {
      const int v = r.m[k];
      bool seen = false;
      for (int t = 0; t < nd; ++t) seen = seen || cn[t] == v;
      if (seen) continue;
      int p = nd++;
      for (; p > 0 && cn[p - 1] > v; --p) cn[p] = cn[p - 1];
      cn[p] = v;
   }
   const double w = nd == 1 ? 1. : (nd == 2 ? 0.5 : 0.25);
#pragma unroll
   for (int c = 0; c < 2; ++c)
   {
      if (fbc && fbc[2 * i + c]) continue;
      double v = 0.;
      bool any = false;
      for (int t = 0; t < nd; ++t)
      {
         if (cbc && cbc[2 * cn[t] + c]) continue;
         const double s = nd == 1 ? xc[2 * cn[t] + c] : __dmul_rn(w, xc[2 * cn[t] + c]);
         v = t == 0 ? s : __dadd_rn(v, s);
         any = true;
      }
      if (any) x[2 * i + c] = __dadd_rn(x[2 * i + c], v);
   }
}

// first Chebyshev step: r = D^-1 (b - t) (t = A x, or null when x = 0);  d = r / theta;  x = d (x0 = 0) or x += d
__global__ void __launch_bounds__(kMgThreads)
mg_cheb_first_kernel(int64_t n2, const double2 *__restrict__ b, const double2 *__restrict__ t, const double2 *__restrict__ dinv,
                     double2 *__restrict__ r, double2 *__restrict__ d, double2 *__restrict__ x, double inv_theta, int xzero)
{
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n2; i += stride)
   {
      double2 ri = b[i];
      if (t)
      {
         const double2 ti = t[i];
         ri.x = __dsub_rn(ri.x, ti.x), ri.y = __dsub_rn(ri.y, ti.y);
      }
      const double2 pi = dinv[i];
      ri.x = __dmul_rn(pi.x, ri.x), ri.y = __dmul_rn(pi.y, ri.y);
      const double2 di = make_double2(__dmul_rn(ri.x, inv_theta), __dmul_rn(ri.y, inv_theta));
      r[i] = ri;
      d[i] = di;
      if (xzero)
         x[i] = di;
      else
      {
         double2 xi = x[i];
         xi.x = __dadd_rn(xi.x, di.x), xi.y = __dadd_rn(xi.y, di.y);
         x[i] = xi;
      }
   }
}

// r -= D^-1 t (t = A d);  d = c1 d + c2 r;  x += d
__global__ void __launch_bounds__(kMgThreads)
mg_cheb_step_kernel(int64_t n2, const double2 *__restrict__ t, const double2 *__restrict__ dinv, double2 *__restrict__ r,
                    double2 *__restrict__ d, double2 *__restrict__ x, double c1, double c2)
{
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 ti = t[i], pi = dinv[i];
      double2 ri = r[i], di = d[i], xi = x[i];
      ri.x = __fma_rn(-pi.x, ti.x, ri.x), ri.y = __fma_rn(-pi.y, ti.y, ri.y);
      di.x = __fma_rn(c1, di.x, __dmul_rn(c2, ri.x)), di.y = __fma_rn(c1, di.y, __dmul_rn(c2, ri.y));
      xi.x = __dadd_rn(xi.x, di.x), xi.y = __dadd_rn(xi.y, di.y);
      r[i] = ri, d[i] = di, x[i] = xi;
   }
}

// x = C b, C dense row-major n x n: one warp per row, lanes over the columns, fixed-tree warp sum
__global__ void __launch_bounds__(kMgThreads)
mg_gemv_kernel(int64_t n, const double *__restrict__ C, const double *__restrict__ b, double *__restrict__ x)
{
   const int64_t row = ((int64_t)blockIdx.x * kMgThreads + threadIdx.x) >> 5;
   const int lane = threadIdx.x & 31;
   if (row >= n) return;
   const double *c = C + row * n;
   double s = 0.;
   for (int64_t j = lane; j < n; j += 32) s = __fma_rn(c[j], b[j], s);
   s = warp_sum(s);
   if (lane == 0) x[row] = s;
}

// dense n x n (n = 2 nnodes) image of a CSR level matrix: one block per node row pair, zero then scatter
__global__ void __launch_bounds__(128)
mg_dense_kernel(int64_t nnodes, const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                const double *__restrict__ val, double *__restrict__ dense)
{
   const int64_t I = blockIdx.x, n = 2 * nnodes;
   double *r0 = dense + 2 * I * n, *r1 = r0 + n;
   for (int64_t j = threadIdx.x; j < n; j += blockDim.x) r0[j] = 0., r1[j] = 0.;
   __syncthreads();
   const int64_t b0 = brp[I];
   const int nb = (int)(brp[I + 1] - b0);
   for (int k = threadIdx.x; k < nb; k += blockDim.x)
   {
      const int64_t J = bcol[b0 + k];
      r0[2 * J] = val[4 * b0 + 2 * k], r0[2 * J + 1] = val[4 * b0 + 2 * k + 1];
      r1[2 * J] = val[4 * b0 + 2 * nb + 2 * k], r1[2 * J + 1] = val[4 * b0 + 2 * nb + 2 * k + 1];
   }
}

// power iteration on D^-1 A: x0 = seeded uniform, normalised; then y = D^-1 A x, x = y / |y|; |y| of the last step
__global__ void __launch_bounds__(kMgThreads) mg_seed_kernel(int64_t n, double *__restrict__ x, ReduceScratch red, double *out)
{
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n; i += stride)
   {
      const double v = hash_uniform((uint64_t)i);
      x[i] = v;
      part = __fma_rn(v, v, part);
   }
   block_reduce_finish<kMgThreads>(part, red, out);
}

__global__ void __launch_bounds__(kMgThreads)
mg_scale_dot_kernel(int64_t n, const double *__restrict__ dinv, const double *__restrict__ t, double *__restrict__ y,
                    ReduceScratch red, double *out)
{
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n; i += stride)
   {
      const double v = __dmul_rn(dinv[i], t[i]);
      y[i] = v;
      part = __fma_rn(v, v, part);
   }
   block_reduce_finish<kMgThreads>(part, red, out);
}

__global__ void __launch_bounds__(kMgThreads)
mg_normalize_kernel(int64_t n, const double *__restrict__ y, const double *__restrict__ nrm2, double *__restrict__ x)
{
   const double s = 1. / sqrt(*nrm2);
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n; i += stride) x[i] = __dmul_rn(y[i], s);
}

// ---- PCG with B = V-cycle: the update kernels that read an explicit z = B r --------------------------------------
// x += alpha d;  r -= alpha A d  (mfem::CGSolver updates x before it tests <B r, r>)
__global__ void __launch_bounds__(kMgThreads)
mg_cg_update_xr_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ d,
                       const double2 *__restrict__ Ad, double2 *__restrict__ x, double2 *__restrict__ r)
{
   if (scal[SC_FLAG] != 0.) return;
   const double alpha = scal[SC_ALPHA];
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 di = d[i], zi = Ad[i];
      double2 xi = x[i], ri = r[i];
      xi.x = __fma_rn(alpha, di.x, xi.x), xi.y = __fma_rn(alpha, di.y, xi.y);
      ri.x = __fma_rn(-alpha, zi.x, ri.x), ri.y = __fma_rn(-alpha, zi.y, ri.y);
      x[i] = xi, r[i] = ri;
   }
}

// partial <z, r> (no-op once the flag is set)
__global__ void __launch_bounds__(kMgThreads)
mg_cg_dot_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ z, const double2 *__restrict__ r,
                 ReduceScratch red, double *__restrict__ out)
{
   if (scal[SC_FLAG] != 0.) return;
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 zi = z[i], ri = r[i];
      part = __fma_rn(zi.x, ri.x, part), part = __fma_rn(zi.y, ri.y, part);
   }
   block_reduce_finish<kMgThreads>(part, red, out);
}

// d = z (init) or d = z + beta d
__global__ void __launch_bounds__(kMgThreads)
mg_cg_update_dir_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ z, double2 *__restrict__ d,
                        int init)
{
   if (!init && scal[SC_FLAG] != 0.) return;
   const double beta = init ? 0. : scal[SC_BETA];
   const int64_t stride = (int64_t)gridDim.x * kMgThreads;
   for (int64_t i = (int64_t)blockIdx.x * kMgThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 zi = z[i];
      if (init)
         d[i] = zi;
      else
      {
         double2 di = d[i];
         di.x = __fma_rn(beta, di.x, zi.x), di.y = __fma_rn(beta, di.y, zi.y);
         d[i] = di;
      }
   }
}

unsigned mg_grid(int64_t n)
{
   const int64_t want = cdiv(n, kMgThreads), cap = (int64_t)devinfo().sm_count * 8;
   return (unsigned)std::max<int64_t>(1, std::min(want, cap));
}

template <typename T>
int mg_alloc(T **p, int64_t count, size_t *bytes)
{
   const size_t b = (size_t)std::max<int64_t>(count, 1) * sizeof(T);
   FEMB_CUDA(cudaMalloc(p, b));
   *bytes += b;
   return 0;
}

}  // namespace
}  // namespace femb

struct femb200_mg
{
   std::vector<femb::MgLevel> lev;  // 0 .. L
   int width = 2;                   // transfer map width (2 pairs, 4 with quad centres)
   int degree = 2;
   double lo_frac = 0.25;
   double *cinv = nullptr;  // [nc x nc]
   double *scal = nullptr;  // [L + 1] power-iteration norms
   int *err = nullptr;
   bool have_values = false, have_inverse = false;
   size_t bytes = 0;
};

namespace femb {
int pa_apply_launch(const femb200_pa *pa, const double *d_x, double *d_y, const double *d_flag, double *d_dot_out,
                    cudaStream_t st, bool accumulate);
int pa_mg_info(const femb200_pa *pa, int *etype, int64_t *nnodes, int64_t *ncells);
const uint8_t *pa_dirichlet_marker(const femb200_pa *pa);
int pa_check_pcoarsening(const femb200_pa *pa, const femb200_plan *coarse, const int32_t *d_map, int width, int *d_err,
                         cudaStream_t st);
int pa_element_galerkin(const femb200_pa *pa, const femb200_plan *coarse, double *d_values, cudaStream_t st);
}  // namespace femb

using namespace femb;

static void mg_free(femb200_mg *mg)
{
   if (!mg) return;
   for (size_t l = 0; l < mg->lev.size(); ++l)
   {
      MgLevel &v = mg->lev[l];
      cudaFree(v.own_values), cudaFree(v.dinv), cudaFree(v.r), cudaFree(v.d), cudaFree(v.t);
      cudaFree(v.b), cudaFree(v.x), cudaFree(v.map), cudaFree(v.slot_fine);
   }
   cudaFree(mg->cinv), cudaFree(mg->scal), cudaFree(mg->err);
   delete mg;
}

extern "C" void femb200_mg_destroy(femb200_mg *mg) { mg_free(mg); }

// Dirichlet marker of a level, read at every launch: femb200_plan_set_dirichlet / femb200_pa_set_dirichlet replace it
static const uint8_t *level_bc(const MgLevel &v) { return v.pa ? pa_dirichlet_marker(v.pa) : v.plan->bc; }

// y = A_l x: the level's SpMV, or the matrix-free apply of level 0
static int mg_apply(const femb200_mg *mg, int l, const double *x, double *y, cudaStream_t st)
{
   const MgLevel &v = mg->lev[l];
   if (v.pa) return pa_apply_launch(v.pa, x, y, nullptr, nullptr, st, false);
   return femb200_spmv(v.plan, v.values, x, y, st);
}

static int mg_create_impl(femb200_mg *mg, int op_kind, const void *fine_op, int nlevels, femb200_plan *const *coarse_plans,
                          const int32_t *const *d_maps, const uint8_t *const *d_coarse_bc, cudaStream_t st)
{
   mg->lev.resize(nlevels + 1);
   for (int l = 0; l <= nlevels; ++l)
   {
      MgLevel &v = mg->lev[l];
      if (l == 0 && op_kind == FEMB200_OP_PA)
      {
         v.pa = static_cast<const femb200_pa *>(fine_op);
         int et = 0;
         int64_t nn = 0, ncell = 0;
         if (int rc = pa_mg_info(v.pa, &et, &nn, &ncell)) return rc;
         FEMB_CHECK(et == FEMB200_P2 || et == FEMB200_Q2,
                    "mg_create: a matrix-free fine level must be P2 or Q2, its first coarse level a p-coarsening (P2 -> P1 "
                    "or Q2 -> Q1 on the same cells)");
         v.nnodes = nn, v.n = 2 * nn;
         continue;
      }
      v.plan = l == 0 ? const_cast<femb200_plan *>(static_cast<const femb200_plan *>(fine_op)) : coarse_plans[l - 1];
      FEMB_CHECK(v.plan, "mg_create: null plan of level %d", l);
      if (l > 0)
      {
         const int want = mg->width == 2 ? FEMB200_P1 : FEMB200_Q1;
         FEMB_CHECK(v.plan->etype == want, "mg_create: coarse level %d is not a %s plan (transfer maps of width %d)", l,
                    want == FEMB200_P1 ? "P1" : "Q1", mg->width);
      }
      v.nnodes = v.plan->nnodes, v.n = 2 * v.nnodes;
   }
   const int64_t nc = mg->lev[nlevels].n;
   FEMB_CHECK(nc <= 16384, "mg_create: the coarsest level has %lld dofs; its dense inverse is limited to 16384",
              (long long)nc);
   if (mg_alloc(&mg->err, 1, &mg->bytes) || mg_alloc(&mg->scal, nlevels + 1, &mg->bytes) ||
       mg_alloc(&mg->cinv, nc * nc, &mg->bytes))
      return 1;
   FEMB_CUDA(cudaMemsetAsync(mg->err, 0, sizeof(int), st));
   const int W = mg->width;
   for (int l = 0; l <= nlevels; ++l)
   {
      MgLevel &v = mg->lev[l];
      if (l > 0)
      {
         if (d_coarse_bc && d_coarse_bc[l - 1])
         {
            if (int rc = femb200_plan_set_dirichlet(v.plan, d_coarse_bc[l - 1], st)) return rc;
         }
         else if (int rc = femb200_plan_set_dirichlet(v.plan, nullptr, st))
            return rc;
         if (mg_alloc(&v.own_values, 4 * v.plan->nnzb, &mg->bytes) || mg_alloc(&v.b, v.n, &mg->bytes) ||
             mg_alloc(&v.x, v.n, &mg->bytes))
            return 1;
         v.values = v.own_values;
      }
      if (l == nlevels) continue;
      if (mg_alloc(&v.dinv, v.n, &mg->bytes) || mg_alloc(&v.r, v.n, &mg->bytes) || mg_alloc(&v.d, v.n, &mg->bytes) ||
          mg_alloc(&v.t, v.n, &mg->bytes))
         return 1;
      const femb200_plan *cp = mg->lev[l + 1].plan;
      const int32_t deg = cp->max_deg;
      FEMB_CHECK(deg <= 32, "mg_create: coarse level %d has a node with %d neighbours (at most 32)", l + 1, deg);
      v.group = deg <= 8 ? 8 : (deg <= 16 ? 16 : 32);
      FEMB_CHECK(d_maps && d_maps[l], "mg_create: null transfer map of level %d", l);
      if (mg_alloc(&v.map, v.nnodes * W, &mg->bytes) || mg_alloc(&v.slot_fine, cp->nnzb, &mg->bytes)) return 1;
      FEMB_CUDA(cudaMemcpyAsync(v.map, d_maps[l], (size_t)v.nnodes * W * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
      FEMB_CUDA(cudaMemsetAsync(v.slot_fine, 0xff, (size_t)cp->nnzb * sizeof(int32_t), st));
      const unsigned g1 = (unsigned)cdiv(v.nnodes, 256), g2 = (unsigned)cdiv(std::max<int64_t>(v.nnodes, cp->nnzb), 256);
      if (W == 2)
      {
         mg_slots_kernel<2><<<g1, 256, 0, st>>>(v.nnodes, v.map, cp->nnodes, cp->brp, cp->bcol, v.slot_fine, mg->err);
         FEMB_LAUNCH_CHECK();
         mg_slots_check_kernel<2><<<g2, 256, 0, st>>>(v.nnodes, v.map, cp->brp, cp->bcol, v.slot_fine, cp->nnzb, mg->err);
      }
      else
      {
         mg_slots_kernel<4><<<g1, 256, 0, st>>>(v.nnodes, v.map, cp->nnodes, cp->brp, cp->bcol, v.slot_fine, mg->err);
         FEMB_LAUNCH_CHECK();
         mg_slots_check_kernel<4><<<g2, 256, 0, st>>>(v.nnodes, v.map, cp->brp, cp->bcol, v.slot_fine, cp->nnzb, mg->err);
      }
      FEMB_LAUNCH_CHECK();
      int herr = 0;
      FEMB_CUDA(cudaMemcpyAsync(&herr, mg->err, sizeof(int), cudaMemcpyDeviceToHost, st));
      FEMB_CUDA(cudaStreamSynchronize(st));
      static const char *what[] = {"", "a coarse node id is out of range",
                                   "a fine node's coarse pair (edge or quad diagonal) is not in the coarse pattern",
                                   "two fine nodes map to the same coarse node, edge or quad",
                                   "a coarse node, edge or quad has no fine node",
                                   "a width-4 map row is none of (a, a, a, a), (a, b, a, b), four distinct nodes"};
      FEMB_CHECK(herr == 0, "mg_create: level %d -> %d is not a nested hierarchy: %s", l, l + 1, what[herr % 6]);
      if (l == 0 && v.pa)
         if (int rc = pa_check_pcoarsening(v.pa, cp, v.map, W, mg->err, st)) return rc;
   }
   return 0;
}

extern "C" int femb200_mg_create_op(int op_kind, const void *fine_op, int nlevels, femb200_plan *const *coarse_plans,
                                    const int32_t *const *d_maps, int map_width, const uint8_t *const *d_coarse_bc,
                                    int degree, double lo_frac, void *stream, femb200_mg **out)
{
   FEMB_CHECK(out && fine_op && nlevels >= 1 && coarse_plans && d_maps, "mg_create: bad argument");
   FEMB_CHECK(op_kind == FEMB200_OP_CSR || op_kind == FEMB200_OP_PA, "mg_create: unknown operator kind %d", op_kind);
   FEMB_CHECK(map_width == 2 || map_width == 4, "mg_create: transfer map width %d (2 or 4)", map_width);
   FEMB_CHECK(degree >= 1 && degree <= kMaxDegree, "mg_create: Chebyshev degree %d outside [1, %d]", degree, kMaxDegree);
   FEMB_CHECK(lo_frac > 0. && lo_frac < 1., "mg_create: lower interval fraction %g outside (0, 1)", lo_frac);
   *out = nullptr;
   femb200_mg *mg = new femb200_mg();
   mg->width = map_width, mg->degree = degree, mg->lo_frac = lo_frac;
   if (int rc = mg_create_impl(mg, op_kind, fine_op, nlevels, coarse_plans, d_maps, d_coarse_bc, as_stream(stream)))
   {
      cudaStreamSynchronize(as_stream(stream));
      mg_free(mg);
      return rc;
   }
   *out = mg;
   return 0;
}

extern "C" int femb200_mg_create(const femb200_plan *fine, int nlevels, femb200_plan *const *coarse_plans,
                                 const int32_t *const *d_maps, const uint8_t *const *d_coarse_bc, int degree,
                                 double lo_frac, void *stream, femb200_mg **out)
{
   return femb200_mg_create_op(FEMB200_OP_CSR, fine, nlevels, coarse_plans, d_maps, 2, d_coarse_bc, degree, lo_frac,
                               stream, out);
}

extern "C" int femb200_mg_sizes(const femb200_mg *mg, int *nlevels, int64_t *ndofs, int64_t *nnz, double *lambda,
                                int64_t *device_bytes)
{
   FEMB_CHECK(mg, "mg_sizes: null handle");
   const int L = (int)mg->lev.size() - 1;
   if (nlevels) *nlevels = L;
   for (int l = 0; l <= L; ++l)
   {
      if (ndofs) ndofs[l] = mg->lev[l].n;
      if (nnz) nnz[l] = mg->lev[l].plan ? 4 * mg->lev[l].plan->nnzb : 0;
      if (lambda) lambda[l] = mg->lev[l].lambda;
   }
   if (device_bytes) *device_bytes = (int64_t)mg->bytes;
   return 0;
}

template <int W>
static void mg_rap_launch(const MgLevel &f, const MgLevel &c, cudaStream_t st)
{
   const femb200_plan *fp = f.plan, *cp = c.plan;
   const unsigned grid = (unsigned)cdiv(cp->nnodes * f.group, kMgThreads);
   switch (f.group)
   {
   case 8:
      mg_rap_kernel<8, W><<<grid, kMgThreads, 0, st>>>(cp->nnodes, cp->brp, cp->bcol, f.slot_fine, fp->brp, fp->bcol,
                                                      f.values, f.map, fp->bc, c.own_values);
      break;
   case 16:
      mg_rap_kernel<16, W><<<grid, kMgThreads, 0, st>>>(cp->nnodes, cp->brp, cp->bcol, f.slot_fine, fp->brp, fp->bcol,
                                                       f.values, f.map, fp->bc, c.own_values);
      break;
   default:
      mg_rap_kernel<32, W><<<grid, kMgThreads, 0, st>>>(cp->nnodes, cp->brp, cp->bcol, f.slot_fine, fp->brp, fp->bcol,
                                                       f.values, f.map, fp->bc, c.own_values);
   }
}

extern "C" int femb200_mg_galerkin(femb200_mg *mg, const double *d_fine_values, int level, void *stream)
{
   FEMB_CHECK(mg, "mg_galerkin: null handle");
   const int L = (int)mg->lev.size() - 1;
   FEMB_CHECK(level >= 0 && level < L, "mg_galerkin: level %d outside [0, %d)", level, L);
   const bool elem = level == 0 && mg->lev[0].pa;  // matrix-free level 0: element Galerkin step
   if (elem)
      FEMB_CHECK(!d_fine_values, "mg_galerkin: the fine level is matrix-free: pass no fine values (NULL)");
   else if (level == 0)
   {
      FEMB_CHECK(d_fine_values, "mg_galerkin: null fine values");
      mg->lev[0].values = d_fine_values;
   }
   FEMB_CHECK(elem || mg->lev[level].values, "mg_galerkin: level %d has no values yet", level);
   const MgLevel &f = mg->lev[level];
   MgLevel &c = mg->lev[level + 1];
   cudaStream_t st = as_stream(stream);
   if (elem)
   {
      if (int rc = pa_element_galerkin(f.pa, c.plan, c.own_values, st)) return rc;
   }
   else
   {
      if (mg->width == 2)
         mg_rap_launch<2>(f, c, st);
      else
         mg_rap_launch<4>(f, c, st);
      FEMB_LAUNCH_CHECK();
   }
   mg->have_inverse = false;
   return femb200_apply_dirichlet(c.plan, c.own_values, 1.0, stream);
}

extern "C" int femb200_mg_setup(femb200_mg *mg, const double *d_fine_values, void *stream)
{
   FEMB_CHECK(mg, "mg_setup: bad argument");
   if (mg->lev[0].pa)
      FEMB_CHECK(!d_fine_values, "mg_setup: the fine level is matrix-free: pass no fine values (NULL)");
   else
      FEMB_CHECK(d_fine_values, "mg_setup: bad argument");
   cudaStream_t st = as_stream(stream);
   const int L = (int)mg->lev.size() - 1;
   for (int l = 0; l < L; ++l)
      if (int rc = femb200_mg_galerkin(mg, d_fine_values, l, stream)) return rc;
   // smoother: D^-1 and the power-iteration estimate of lambda_max(D^-1 A) on every level but the coarsest
   for (int l = 0; l < L; ++l)
   {
      MgLevel &v = mg->lev[l];
      if (v.pa)
      {  // carries diag on the constrained dofs (femb200_pa_set_dirichlet), as the assembled diagonal does
         if (int rc = femb200_pa_diagonal(v.pa, v.dinv, stream)) return rc;
      }
      else if (int rc = femb200_extract_diagonal(v.plan, v.values, v.dinv, stream))
         return rc;
      if (int rc = femb200_jacobi_setup(v.n, v.dinv, v.dinv, stream)) return rc;
      // the fused-reduction scratch is taken right before every reducing kernel: an SpMV launch in between may grow
      // (reallocate) the scratch of the stream
      const unsigned grid = mg_grid(v.n);
      ReduceScratch red;
      if (int rc = reduce_scratch(grid, st, &red)) return rc;
      mg_seed_kernel<<<grid, kMgThreads, 0, st>>>(v.n, v.t, red, mg->scal + l);
      FEMB_LAUNCH_CHECK();
      mg_normalize_kernel<<<grid, kMgThreads, 0, st>>>(v.n, v.t, mg->scal + l, v.d);
      FEMB_LAUNCH_CHECK();
      for (int it = 0; it < kPowerIters; ++it)
      {
         if (int rc = mg_apply(mg, l, v.d, v.t, st)) return rc;
         if (int rc = reduce_scratch(grid, st, &red)) return rc;
         mg_scale_dot_kernel<<<grid, kMgThreads, 0, st>>>(v.n, v.dinv, v.t, v.r, red, mg->scal + l);
         FEMB_LAUNCH_CHECK();
         mg_normalize_kernel<<<grid, kMgThreads, 0, st>>>(v.n, v.r, mg->scal + l, v.d);
         FEMB_LAUNCH_CHECK();
      }
   }
   std::vector<double> h(L + 1, 0.);
   FEMB_CUDA(cudaMemcpyAsync(h.data(), mg->scal, sizeof(double) * (L + 1), cudaMemcpyDeviceToHost, st));
   FEMB_CUDA(cudaStreamSynchronize(st));
   for (int l = 0; l < L; ++l)
   {
      MgLevel &v = mg->lev[l];
      FEMB_CHECK(h[l] > 0. && isfinite(h[l]), "mg_setup: the power iteration of level %d gave |D^-1 A x|^2 = %g", l,
                 h[l]);
      v.lambda = 1.1 * sqrt(h[l]);
      // Chebyshev on [lo lambda, lambda]: theta = centre, delta = half width, sigma = theta / delta
      const double a = mg->lo_frac * v.lambda, bb = v.lambda;
      const double theta = 0.5 * (bb + a), delta = 0.5 * (bb - a), sigma = theta / delta;
      double rho = 1. / sigma;
      v.inv_theta = 1. / theta;
      for (int s = 1; s < mg->degree; ++s)
      {
         const double rho_n = 1. / (2. * sigma - rho);
         v.c1[s] = rho_n * rho, v.c2[s] = 2. * rho_n / delta;
         rho = rho_n;
      }
   }
   mg->have_values = true;
   mg->have_inverse = false;
   return 0;
}

extern "C" int femb200_mg_level_values(const femb200_mg *mg, int level, double *d_out, void *stream)
{
   FEMB_CHECK(mg && d_out, "mg_level_values: bad argument");
   const int L = (int)mg->lev.size() - 1;
   FEMB_CHECK(level >= 1 && level <= L, "mg_level_values: level %d outside [1, %d]", level, L);
   const MgLevel &v = mg->lev[level];
   FEMB_CUDA(cudaMemcpyAsync(d_out, v.own_values, sizeof(double) * 4 * v.plan->nnzb, cudaMemcpyDeviceToDevice,
                             as_stream(stream)));
   return 0;
}

extern "C" int femb200_mg_coarse_matrix(const femb200_mg *mg, double *d_dense, void *stream)
{
   FEMB_CHECK(mg && d_dense, "mg_coarse_matrix: bad argument");
   const MgLevel &v = mg->lev.back();
   mg_dense_kernel<<<(unsigned)v.nnodes, 128, 0, as_stream(stream)>>>(v.nnodes, v.plan->brp, v.plan->bcol, v.values, d_dense);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_mg_set_coarse_inverse(femb200_mg *mg, const double *d_inv, void *stream)
{
   FEMB_CHECK(mg && d_inv, "mg_set_coarse_inverse: bad argument");
   const int64_t nc = mg->lev.back().n;
   FEMB_CUDA(cudaMemcpyAsync(mg->cinv, d_inv, sizeof(double) * nc * nc, cudaMemcpyDeviceToDevice, as_stream(stream)));
   mg->have_inverse = true;
   return 0;
}

extern "C" int femb200_mg_restrict(const femb200_mg *mg, int level, const double *d_b, const double *d_t, double *d_bc,
                                   void *stream)
{
   FEMB_CHECK(mg && d_b && d_bc, "mg_restrict: bad argument");
   const int L = (int)mg->lev.size() - 1;
   FEMB_CHECK(level >= 0 && level < L, "mg_restrict: level %d outside [0, %d)", level, L);
   const MgLevel &f = mg->lev[level], &c = mg->lev[level + 1];
   const unsigned grid = (unsigned)cdiv(c.nnodes, kMgThreads);
   const auto b = reinterpret_cast<const double2 *>(d_b), t = reinterpret_cast<const double2 *>(d_t);
   const auto out = reinterpret_cast<double2 *>(d_bc);
   if (mg->width == 2)
      mg_restrict_kernel<2><<<grid, kMgThreads, 0, as_stream(stream)>>>(c.nnodes, c.plan->brp, f.slot_fine, f.map,
                                                                         level_bc(f), level_bc(c), b, t, out);
   else
      mg_restrict_kernel<4><<<grid, kMgThreads, 0, as_stream(stream)>>>(c.nnodes, c.plan->brp, f.slot_fine, f.map,
                                                                         level_bc(f), level_bc(c), b, t, out);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_mg_prolong(const femb200_mg *mg, int level, const double *d_xc, double *d_x, void *stream)
{
   FEMB_CHECK(mg && d_xc && d_x, "mg_prolong: bad argument");
   const int L = (int)mg->lev.size() - 1;
   FEMB_CHECK(level >= 0 && level < L, "mg_prolong: level %d outside [0, %d)", level, L);
   const MgLevel &f = mg->lev[level], &c = mg->lev[level + 1];
   const unsigned grid = (unsigned)cdiv(f.nnodes, kMgThreads);
   if (mg->width == 2)
      mg_prolong_kernel<2><<<grid, kMgThreads, 0, as_stream(stream)>>>(f.nnodes, f.map, level_bc(f), level_bc(c), d_xc,
                                                                        d_x);
   else
      mg_prolong_kernel<4><<<grid, kMgThreads, 0, as_stream(stream)>>>(f.nnodes, f.map, level_bc(f), level_bc(c), d_xc,
                                                                        d_x);
   FEMB_LAUNCH_CHECK();
   return 0;
}

namespace femb {
namespace {

// Optional per-launch timing of a V-cycle (femb200_mg_vcycle_timed): an event after every launch; the time between
// consecutive events goes to the (level, kind) of the launch that ends it, launch gaps included.
enum
{
   MG_T_SPMV = 0,
   MG_T_CHEB = 1,
   MG_T_RESTRICT = 2,
   MG_T_PROLONG = 3,
   MG_T_COARSE = 4,
   MG_T_KINDS = 5
};
struct MgTimer
{
   std::vector<cudaEvent_t> ev;
   std::vector<int> slot;  // level * MG_T_KINDS + kind of the launch that ends at ev[k] (k >= 1)
   int mark(int level, int kind, cudaStream_t st)
   {
      cudaEvent_t e;
      FEMB_CUDA(cudaEventCreate(&e));
      ev.push_back(e);
      slot.push_back(level * MG_T_KINDS + kind);
      FEMB_CUDA(cudaEventRecord(e, st));
      return 0;
   }
   ~MgTimer()
   {
      for (cudaEvent_t e : ev) cudaEventDestroy(e);
   }
};
#define MG_MARK(tm, level, kind)                                             \
   do                                                                       \
   {                                                                        \
      if (tm)                                                               \
         if (int rc__ = (tm)->mark((level), (kind), st)) return rc__;       \
   } while (0)

int mg_smooth(const femb200_mg *mg, int l, const double *b, double *x, bool xzero, cudaStream_t st, MgTimer *tm)
{
   const MgLevel &v = mg->lev[l];
   const int64_t n2 = v.n / 2;
   const unsigned grid = mg_grid(n2);
   if (!xzero)
   {
      if (int rc = mg_apply(mg, l, x, v.t, st)) return rc;
      MG_MARK(tm, l, MG_T_SPMV);
   }
   mg_cheb_first_kernel<<<grid, kMgThreads, 0, st>>>(
       n2, reinterpret_cast<const double2 *>(b), xzero ? nullptr : reinterpret_cast<const double2 *>(v.t),
       reinterpret_cast<const double2 *>(v.dinv), reinterpret_cast<double2 *>(v.r), reinterpret_cast<double2 *>(v.d),
       reinterpret_cast<double2 *>(x), v.inv_theta, xzero ? 1 : 0);
   FEMB_LAUNCH_CHECK();
   MG_MARK(tm, l, MG_T_CHEB);
   for (int s = 1; s < mg->degree; ++s)
   {
      if (int rc = mg_apply(mg, l, v.d, v.t, st)) return rc;
      MG_MARK(tm, l, MG_T_SPMV);
      mg_cheb_step_kernel<<<grid, kMgThreads, 0, st>>>(n2, reinterpret_cast<const double2 *>(v.t),
                                                       reinterpret_cast<const double2 *>(v.dinv), reinterpret_cast<double2 *>(v.r),
                                                       reinterpret_cast<double2 *>(v.d), reinterpret_cast<double2 *>(x),
                                                       v.c1[s], v.c2[s]);
      FEMB_LAUNCH_CHECK();
      MG_MARK(tm, l, MG_T_CHEB);
   }
   return 0;
}

int mg_vcycle_level(const femb200_mg *mg, int l, const double *b, double *x, cudaStream_t st, MgTimer *tm)
{
   const int L = (int)mg->lev.size() - 1;
   const MgLevel &v = mg->lev[l];
   if (l == L)
   {
      mg_gemv_kernel<<<(unsigned)cdiv(v.n * 32, kMgThreads), kMgThreads, 0, st>>>(v.n, mg->cinv, b, x);
      FEMB_LAUNCH_CHECK();
      MG_MARK(tm, l, MG_T_COARSE);
      return 0;
   }
   const MgLevel &c = mg->lev[l + 1];
   if (int rc = mg_smooth(mg, l, b, x, true, st, tm)) return rc;
   if (int rc = mg_apply(mg, l, x, v.t, st)) return rc;
   MG_MARK(tm, l, MG_T_SPMV);
   if (int rc = femb200_mg_restrict(mg, l, b, v.t, c.b, st)) return rc;
   MG_MARK(tm, l, MG_T_RESTRICT);
   if (int rc = mg_vcycle_level(mg, l + 1, c.b, c.x, st, tm)) return rc;
   if (int rc = femb200_mg_prolong(mg, l, c.x, x, st)) return rc;
   MG_MARK(tm, l, MG_T_PROLONG);
   return mg_smooth(mg, l, b, x, false, st, tm);
}

int mg_vcycle_check(const femb200_mg *mg, const double *d_r, const double *d_z)
{
   FEMB_CHECK(mg && d_r && d_z, "mg_vcycle: bad argument");
   // level 0 reads r (its right-hand side) again after it has written z
   FEMB_CHECK(d_r != d_z, "mg_vcycle: r and z must be different vectors");
   FEMB_CHECK(mg->have_values, "mg_vcycle: run femb200_mg_setup first");
   FEMB_CHECK(mg->have_inverse, "mg_vcycle: no coarse inverse for the current coarse operator (femb200_mg_set_coarse_inverse)");
   return 0;
}

}  // namespace
}  // namespace femb

extern "C" int femb200_mg_vcycle(femb200_mg *mg, const double *d_r, double *d_z, void *stream)
{
   if (int rc = mg_vcycle_check(mg, d_r, d_z)) return rc;
   return mg_vcycle_level(mg, 0, d_r, d_z, as_stream(stream), nullptr);
}

extern "C" int femb200_mg_vcycle_timed(femb200_mg *mg, const double *d_r, double *d_z, double *ms, void *stream)
{
   if (int rc = mg_vcycle_check(mg, d_r, d_z)) return rc;
   FEMB_CHECK(ms, "mg_vcycle_timed: null output");
   cudaStream_t st = as_stream(stream);
   const int L = (int)mg->lev.size() - 1;
   MgTimer tm;
   if (int rc = tm.mark(0, 0, st)) return rc;
   if (int rc = mg_vcycle_level(mg, 0, d_r, d_z, st, &tm)) return rc;
   FEMB_CUDA(cudaEventSynchronize(tm.ev.back()));
   for (int k = 0; k < (L + 1) * MG_T_KINDS; ++k) ms[k] = 0.;
   for (size_t k = 1; k < tm.ev.size(); ++k)
   {
      float t = 0.f;
      FEMB_CUDA(cudaEventElapsedTime(&t, tm.ev[k - 1], tm.ev[k]));
      ms[tm.slot[k]] += t;
   }
   return 0;
}

extern "C" int femb200_pcg_mg(femb200_mg *mg, const double *d_b, double *d_x, double rtol, double atol, int maxit,
                              int check_every, double *d_work, int *iters, double *final_norm, int *converged, void *stream)
{
   FEMB_CHECK(mg && d_b && d_x && d_work && maxit >= 0, "pcg_mg: bad argument");
   FEMB_CHECK(mg->have_values && mg->have_inverse, "pcg_mg: run femb200_mg_setup and set the coarse inverse first");
   cudaStream_t st = as_stream(stream);
   const MgLevel &f = mg->lev[0];
   const int64_t n = f.n, n2 = n / 2;
   double *r = d_work, *d = d_work + n, *z = d_work + 2 * n, *Ad = d_work + 3 * n, *scal = d_work + 4 * n;
   RowRange rr{0, 0, {0, 0}, 0};
   if (f.plan)
      if (int rc = plan_row_range(f.plan, 0, f.nnodes, &rr)) return rc;
   const unsigned grid = mg_grid(n2);
   auto apply = [&]() -> int {  // Ad = A d with the fused <d, A d> (SpMV or matrix-free apply)
      if (int rc = f.pa ? pa_apply_launch(f.pa, d, Ad, scal + SC_FLAG, scal + SC_RED_DEN, st, false)
                        : spmv_launch(f.plan, rr, f.values, d, Ad, scal + SC_FLAG, scal + SC_RED_DEN, false, st))
         return rc;
      return femb200_cg_scalar_step(scal, 1, st);
   };
   auto precond_dot = [&](int red_slot) -> int {
      if (int rc = femb200_mg_vcycle(mg, r, z, st)) return rc;
      // taken here, not once before the loop: the SpMV launches of the V-cycle and of apply() may grow (reallocate)
      // the fused-reduction scratch of the stream
      ReduceScratch red;
      if (int rc = reduce_scratch(grid, st, &red)) return rc;
      mg_cg_dot_kernel<<<grid, kMgThreads, 0, st>>>(n2, scal, reinterpret_cast<const double2 *>(z),
                                                    reinterpret_cast<const double2 *>(r), red, scal + red_slot);
      FEMB_LAUNCH_CHECK();
      return 0;
   };
   if (int rc = femb200_cg_set_tolerances(scal, rtol, atol, st)) return rc;
   FEMB_CUDA(cudaMemsetAsync(d_x, 0, sizeof(double) * n, st));
   FEMB_CUDA(cudaMemcpyAsync(r, d_b, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
   if (int rc = precond_dot(SC_RED_NOM)) return rc;
   mg_cg_update_dir_kernel<<<grid, kMgThreads, 0, st>>>(n2, scal, reinterpret_cast<const double2 *>(z),
                                                        reinterpret_cast<double2 *>(d), 1);
   FEMB_LAUNCH_CHECK();
   if (int rc = femb200_cg_scalar_step(scal, 0, st)) return rc;
   if (int rc = apply()) return rc;
   const int every = check_every > 0 ? check_every : 1;
   double hs[SC_COUNT];
   for (int i = 1; i <= maxit; ++i)
   {
      mg_cg_update_xr_kernel<<<grid, kMgThreads, 0, st>>>(n2, scal, reinterpret_cast<const double2 *>(d),
                                                          reinterpret_cast<const double2 *>(Ad), reinterpret_cast<double2 *>(d_x),
                                                          reinterpret_cast<double2 *>(r));
      FEMB_LAUNCH_CHECK();
      if (int rc = precond_dot(SC_RED_BETA)) return rc;
      if (int rc = femb200_cg_scalar_step(scal, 2, st)) return rc;
      if (i == maxit) break;
      mg_cg_update_dir_kernel<<<grid, kMgThreads, 0, st>>>(n2, scal, reinterpret_cast<const double2 *>(z),
                                                           reinterpret_cast<double2 *>(d), 0);
      FEMB_LAUNCH_CHECK();
      if (int rc = apply()) return rc;
      if (i % every == 0)
      {
         FEMB_CUDA(cudaMemcpyAsync(hs, scal, sizeof(hs), cudaMemcpyDeviceToHost, st));
         FEMB_CUDA(cudaStreamSynchronize(st));
         if (hs[SC_FLAG] != 0.) break;
      }
   }
   FEMB_CUDA(cudaMemcpyAsync(hs, scal, sizeof(hs), cudaMemcpyDeviceToHost, st));
   FEMB_CUDA(cudaStreamSynchronize(st));
   const bool conv = hs[SC_FLAG] == 1.;
   if (converged) *converged = conv ? 1 : 0;
   if (iters) *iters = (conv || hs[SC_FLAG] == 2.) ? (int)hs[SC_ITERS] : maxit;
   if (final_norm) *final_norm = sqrt(hs[SC_FINAL] > 0. ? hs[SC_FINAL] : 0.);
   return 0;
}
