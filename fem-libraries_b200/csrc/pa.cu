// pa.cu -- partial assembly: matrix-free apply of the elasticity operator.
//
// Role in the reference: mfem BilinearFormIntegrator::AssemblePA / AddMultPA.  The
// reference does not exercise them (its integrator is a NonlinearFormIntegrator,
// M.cc:559,639; partial assembly is only discussed at doc.tex:1445-1449), so the
// contract is SURVEY.md A.9:  y_e = sum_q w_q |det J_q| B_q (D (B_q^t x_e)).
//
// "AssemblePA" (pa_create) builds, once:
//  * a cell order: cells sorted by the Morton code of their centroid, cut into TILES of CT
//    consecutive cells (compact 2-D patches on any mesh with spatial locality);
//  * per tile the sorted list of its unique nodes, the cell -> local node map (16-bit) and its
//    transpose (local node -> the (cell, local dof) pairs that touch it);
//  * per cell (tile order) the straight-sided geometry (nv vertices) and the Lame pair:
//    10 doubles (Q2) / 8 doubles (triangles); J_q is rebuilt per quadrature point (bilinear /
//    affine, a handful of FMAs), which is fewer bytes than storing (J^-1, w) per point.
// "AddMultPA" (pa_apply): one CTA per tile, one thread per cell.  The tile's x values are staged in
// shared memory once (coalesced runs of consecutive nodes), every cell computes its element
// product (sum-factorised for Q2: 1-D 3x3 tables) into a shared E-vector, then one thread per
// tile node sums the contributions of the tile's cells.  Nodes interior to a tile (the vast
// majority) are written with one plain 16-byte store; only nodes on a tile boundary use
// red.global.add.f64 into entries zeroed by a small pre-kernel (compact list built at setup).
// Dirichlet dofs are handled like the assembled operator (rows/cols zeroed, diag on the
// diagonal) through a per-cell bit mask of constrained local dofs.
#include <algorithm>
#include <cub/block/block_discontinuity.cuh>
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>

#include "constitutive.cuh"
#include "element.cuh"
#include "plan.cuh"
#include "reduce.cuh"
#include "tma.cuh"

struct femb200_pa
{
   int etype = 0, nd = 0, nv = 0;
   int64_t nnodes = 0, ncells = 0;
   const int32_t *dofmap = nullptr;  // borrowed
   int ct = 0;                       // cells per tile
   int64_t ntiles = 0;
   int max_uniq = 0;                 // largest number of unique nodes in a tile
   int32_t *cperm = nullptr;         // [ncells] tile order -> caller's cell index
   double *geo = nullptr;            // [ncells][2 nv + 2]: vertices, lambda, mu (tile order)
   int32_t *tcount = nullptr;        // [ntiles] unique nodes of the tile
   int32_t *tnodes = nullptr;        // [ntiles][ct nd] global node of local node k; bit 31: shared with another tile
   uint16_t *tptr = nullptr;         // [ntiles][ct nd + 8]: [0] = unique nodes, [1 + k] = first entry of node k in trefs
   uint16_t *trefs = nullptr;        // [ntiles][nd][ct] position of (cell in tile, a) in the node-sorted E-vector
   uint16_t *lidx = nullptr;         // [ntiles][nd][ct] local node of (cell in tile, a)
   int32_t *shared_nodes = nullptr;  // nodes touched by more than one tile
   int32_t nshared = 0;
   uint32_t *cmask = nullptr;        // [ncells] constrained local dofs (bit 2a+i), tile order, or null
   uint8_t *bc = nullptr;            // [2 nnodes] or null
   int32_t *bc_dofs = nullptr;       // compact list of constrained dofs
   int32_t nbc = 0;
   double diag = 1.0;
   size_t bytes = 0;
};

#ifndef PA_EXP
#define PA_EXP 0
#endif

namespace femb {

constexpr int kPaThreads = 128;  // = cells per tile

// ---- setup: cell order --------------------------------------------------------------
__global__ void pa_centroid_kernel(int64_t ncells, int nv, const int32_t *__restrict__ xdofmap,
                                   const double *__restrict__ x, int xs, float *__restrict__ cx, float *__restrict__ cy)
{
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   double sx = 0., sy = 0.;
   for (int v = 0; v < nv; ++v)
   {
      const int64_t n = xdofmap[e * nv + v];
      sx += x[n * xs], sy += x[n * xs + 1];
   }
   cx[e] = (float)(sx / nv), cy[e] = (float)(sy / nv);
}

__device__ __forceinline__ uint32_t spread16(uint32_t v)
{
   v &= 0xffffu;
   v = (v | (v << 8)) & 0x00ff00ffu;
   v = (v | (v << 4)) & 0x0f0f0f0fu;
   v = (v | (v << 2)) & 0x33333333u;
   v = (v | (v << 1)) & 0x55555555u;
   return v;
}

// bb = (min x, max x, min y, max y) of the centroids
__global__ void pa_morton_kernel(int64_t ncells, const float *__restrict__ cx, const float *__restrict__ cy,
                                 const float *__restrict__ bb, uint32_t *__restrict__ key, int32_t *__restrict__ id)
{
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   const float sx = bb[1] > bb[0] ? 65535.f / (bb[1] - bb[0]) : 0.f, sy = bb[3] > bb[2] ? 65535.f / (bb[3] - bb[2]) : 0.f;
   const uint32_t qx = (uint32_t)fminf(fmaxf((cx[e] - bb[0]) * sx, 0.f), 65535.f);
   const uint32_t qy = (uint32_t)fminf(fmaxf((cy[e] - bb[2]) * sy, 0.f), 65535.f);
   key[e] = spread16(qx) | (spread16(qy) << 1);
   id[e] = (int32_t)e;
}

// ---- setup: per-tile node lists -------------------------------------------------------
// One CTA per tile sorts the (node, a * CT + t) pairs of its cells by node: the heads of the runs
// are the tile's unique nodes (ascending); the sorted position of a pair is where the cell's
// contribution is stored, so that the contributions to one node are contiguous.
template <int ND, int CT>
__global__ void __launch_bounds__(CT)
pa_tile_build_kernel(int64_t ncells, int64_t nnodes, int end_bit, const int32_t *__restrict__ dofmap,
                     const int32_t *__restrict__ cperm, int32_t *__restrict__ tnodes, uint16_t *__restrict__ tptr,
                     uint16_t *__restrict__ trefs, uint16_t *__restrict__ lidx, int32_t *__restrict__ tcount,
                     int32_t *__restrict__ ntouch)
{
   using Sort = cub::BlockRadixSort<uint32_t, CT, ND, uint16_t>;
   using Disc = cub::BlockDiscontinuity<uint32_t, CT>;
   using Scan = cub::BlockScan<int, CT>;
   __shared__ union
   {
      typename Sort::TempStorage sort;
      typename Disc::TempStorage disc;
      typename Scan::TempStorage scan;
   } tmp;
   constexpr int S = CT * ND;
   const int64_t tile = blockIdx.x;
   const int t = threadIdx.x;
   const int64_t e = tile * CT + t;
   const uint32_t none = (uint32_t)nnodes;
   uint32_t key[ND];
   uint16_t val[ND];
   const int64_t row = e < ncells ? (int64_t)cperm[e] * ND : 0;
#pragma unroll
   for (int a = 0; a < ND; ++a)
   {
      key[a] = e < ncells ? (uint32_t)dofmap[row + a] : none;
      val[a] = (uint16_t)(a * CT + t);
   }
   Sort(tmp.sort).Sort(key, val, 0, end_bit);
   __syncthreads();
   int flag[ND];
   Disc(tmp.disc).FlagHeads(flag, key, cub::Inequality());
   __syncthreads();
   int cnt = 0;
#pragma unroll
   for (int j = 0; j < ND; ++j)
   {
      if (key[j] == none) flag[j] = 0;
      cnt += flag[j];
   }
   int lid, total;
   Scan(tmp.scan).ExclusiveSum(cnt, lid, total);
   lid -= 1;  // index of the run that is open when this thread's items start
   const int64_t base = tile * S;
   uint16_t *tp = tptr + tile * (S + 8) + 1;
#pragma unroll
   for (int j = 0; j < ND; ++j)
   {
      if (key[j] == none) continue;
      const int pos = t * ND + j;
      if (flag[j])
      {
         ++lid;
         tnodes[base + lid] = (int32_t)key[j];
         tp[lid] = (uint16_t)pos;
         atomicAdd(ntouch + key[j], 1);
      }
      trefs[base + val[j]] = (uint16_t)pos;
      lidx[base + val[j]] = (uint16_t)lid;
   }
   if (t == 0)
   {
      const int64_t left = ncells - tile * CT;
      tp[total] = (uint16_t)((left < CT ? (int)left : CT) * ND);
      tp[-1] = (uint16_t)total;
      tcount[tile] = total;
   }
}

__global__ void pa_tile_flag_kernel(int64_t ntiles, int S, const int32_t *__restrict__ tcount,
                                    const int32_t *__restrict__ ntouch, int32_t *__restrict__ tnodes)
{
   const int64_t tile = blockIdx.x;
   const int n = tcount[tile];
   for (int k = threadIdx.x; k < n; k += blockDim.x)
   {
      const int32_t node = tnodes[tile * S + k];
      if (ntouch[node] > 1) tnodes[tile * S + k] = node | (int32_t)0x80000000;
   }
}

__global__ void pa_shared_list_kernel(int64_t nnodes, const int32_t *__restrict__ ntouch, int32_t *__restrict__ list,
                                      int32_t *__restrict__ count)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= nnodes || ntouch[i] <= 1) return;
   const int32_t p = atomicAdd(count, 1);
   if (list) list[p] = (int32_t)i;
}

// ---- setup: per-cell data in tile order ----------------------------------------------
template <int ET>
__global__ void pa_setup_kernel(int64_t ncells, const int32_t *__restrict__ cperm, const int32_t *__restrict__ xdofmap,
                                const double *__restrict__ x, int xs, const double *__restrict__ E, LameCoef lc,
                                double *__restrict__ geo)
{
   constexpr int nv = Elem<ET>::nv, W = 2 * nv + 2;
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   const int64_t src = cperm[e];
   // tile-major, then structure of arrays: pair k of cell t of a tile at ((tile * W/2 + k) * CT + t): the apply
   // kernel reads its W/2 pairs with coalesced 16-byte loads (no shared-memory stage for the geometry)
   double2 *g = reinterpret_cast<double2 *>(geo) + (e / kPaThreads) * (W / 2) * kPaThreads + (e % kPaThreads);
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const int64_t n = xdofmap[src * nv + v];
      g[v * kPaThreads] = make_double2(x[n * xs], x[n * xs + 1]);
   }
   g[nv * kPaThreads] = make_double2(E[src] * lc.c2, E[src] * lc.c3);  // lambda, mu (M.cc:1093-1098)
}

__global__ void pa_cmask_kernel(int64_t ncells, int nd, const int32_t *__restrict__ cperm,
                                const int32_t *__restrict__ dofmap, const uint8_t *__restrict__ bc,
                                uint32_t *__restrict__ cmask)
{
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   const int64_t src = cperm[e];
   uint32_t m = 0;
   for (int a = 0; a < nd; ++a)
   {
      const int64_t n = dofmap[src * nd + a];
      if (bc[2 * n]) m |= 1u << (2 * a);
      if (bc[2 * n + 1]) m |= 1u << (2 * a + 1);
   }
   cmask[e] = m;
}

__global__ void pa_bc_list_kernel(int64_t ndofs, const uint8_t *__restrict__ bc, int32_t *__restrict__ list,
                                  int32_t *__restrict__ count)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= ndofs || !bc[i]) return;
   const int32_t p = atomicAdd(count, 1);
   if (list) list[p] = (int32_t)i;
}

// stress at one point: sg = w D (exx, eyy, gxy), Hooke (M.cc:873-881)
__device__ __forceinline__ void hooke_stress(double lam, double mu, double w, double exx, double eyy, double gxy,
                                             double &sxx, double &syy, double &sxy)
{
   const double tr = lam * (exx + eyy);
   sxx = w * (tr + 2. * mu * exx);
   syy = w * (tr + 2. * mu * eyy);
   sxy = w * (mu * gxy);
}

// element-local product ye = K_e xe for triangles: generic loop over the points
template <int ET>
__device__ __forceinline__ void local_apply_tri(const double *g, const double *ux, const double *uy, double *yx,
                                                double *yy)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq;
   double xv[nv][2];
#pragma unroll
   for (int v = 0; v < nv; ++v) xv[v][0] = g[2 * v], xv[v][1] = g[2 * v + 1];
   const double lam = g[2 * nv], mu = g[2 * nv + 1];
#pragma unroll
   for (int a = 0; a < nd; ++a) yx[a] = yy[a] = 0.;
#pragma unroll
   for (int q = 0; q < nq; ++q)
   {
      double G[nd][2], phi[nv];
      const double w = qp_geometry<ET>(xv, q, G, phi);
      double exx = 0., eyy = 0., gxy = 0.;
#pragma unroll
      for (int a = 0; a < nd; ++a)
      {
         exx += G[a][0] * ux[a];
         eyy += G[a][1] * uy[a];
         gxy += G[a][1] * ux[a] + G[a][0] * uy[a];
      }
      double sxx, syy, sxy;
      hooke_stress(lam, mu, w, exx, eyy, gxy, sxx, syy, sxy);
#pragma unroll
      for (int a = 0; a < nd; ++a)
      {
         yx[a] += G[a][0] * sxx + G[a][1] * sxy;
         yy[a] += G[a][1] * syy + G[a][0] * sxy;
      }
   }
}

// Q2: sum factorisation with the 1-D tables of the three Lagrange (GLL) basis functions at the
// three Gauss points t0 < 1/2 < t2.  The tables are
//    B  = [b0 b1 b2; 0 1 0; b2 b1 b0]        dB = [d0 d1 d2; -1 0 1; -d2 -d1 -d0]
// (the middle Gauss point is the middle node), which the contractions below exploit.
namespace q2 {
constexpr double s = 0.7745966692414834;
constexpr double t = 0.5 * (1. - s);
constexpr double b0 = 2. * (t - 0.5) * (t - 1.), b1 = 4. * t * (1. - t), b2 = 2. * t * (t - 0.5);
constexpr double d0 = 4. * t - 3., d1 = 4. - 8. * t, d2 = 4. * t - 1.;
// values at the three points of  sum_i B[q][i] u_i  and  sum_i dB[q][i] u_i
__device__ __forceinline__ void interp(double u0, double u1, double u2, double *v)
{
   v[0] = b0 * u0 + b1 * u1 + b2 * u2;
   v[1] = u1;
   v[2] = b2 * u0 + b1 * u1 + b0 * u2;
}
__device__ __forceinline__ void deriv(double u0, double u1, double u2, double *v)
{
   v[0] = d0 * u0 + d1 * u1 + d2 * u2;
   v[1] = u2 - u0;
   v[2] = -d2 * u0 - d1 * u1 - d0 * u2;
}
// transposes: out_i = sum_q B[q][i] a_q,  out_i = sum_q dB[q][i] a_q
__device__ __forceinline__ void interp_t(double a0, double a1, double a2, double *v)
{
   v[0] = b0 * a0 + b2 * a2;
   v[1] = b1 * (a0 + a2) + a1;
   v[2] = b2 * a0 + b0 * a2;
}
__device__ __forceinline__ void deriv_t_add(double a0, double a1, double a2, double *v)
{
   v[0] += d0 * a0 - a1 - d2 * a2;
   v[1] += d1 * (a0 - a2);
   v[2] += d2 * a0 + a1 - d0 * a2;
}
}  // namespace q2

// 1 / d to ~1 ulp: hardware seed + two Newton steps (no slow-path call)
__device__ __forceinline__ double fast_rcp(double d)
{
   double x;
   asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
   x = fma(fma(-d, x, 1.), x, x);
   x = fma(fma(-d, x, 1.), x, x);
   return x;
}

__device__ __forceinline__ void local_apply_q2(const double *g, const double *ux, const double *uy, double *yx,
                                               double *yy)
{
   const double xq[3] = {q2::t, 0.5, 1. - q2::t};
   const double wq[3] = {5. / 18., 8. / 18., 5. / 18.};
   const double lam = g[8], mu = g[9];
   // reference gradients at the 9 points: a[3 qy + qx] = (dux/dxi, dux/deta, duy/dxi, duy/deta)
   double a[9][4];
#pragma unroll
   for (int c = 0; c < 2; ++c)
   {
      const double *u = c ? uy : ux;
      double t0[3][3], t1[3][3];  // [j][qx]: values / xi-derivatives along node row j
#pragma unroll
      for (int j = 0; j < 3; ++j)
      {
         q2::interp(u[3 * j], u[3 * j + 1], u[3 * j + 2], t0[j]);
         q2::deriv(u[3 * j], u[3 * j + 1], u[3 * j + 2], t1[j]);
      }
#pragma unroll
      for (int qx = 0; qx < 3; ++qx)
      {
         double v[3], w[3];
         q2::interp(t1[0][qx], t1[1][qx], t1[2][qx], v);  // d/dxi at (qx, qy = 0..2)
         q2::deriv(t0[0][qx], t0[1][qx], t0[2][qx], w);   // d/deta
#pragma unroll
         for (int qy = 0; qy < 3; ++qy) a[3 * qy + qx][2 * c] = v[qy], a[3 * qy + qx][2 * c + 1] = w[qy];
      }
   }
   // point work: a[q] <- (px0, px1, py0, py1) = adj(J) (w / |det|) sigma(adj(J)^t grad_ref u)
   const double ax = g[2] - g[0], bx = g[6] - g[4], cx = g[4] - g[0], dx = g[6] - g[2];
   const double ay = g[3] - g[1], by = g[7] - g[5], cy = g[5] - g[1], dy = g[7] - g[3];
#pragma unroll
   for (int qy = 0; qy < 3; ++qy)
#pragma unroll
      for (int qx = 0; qx < 3; ++qx)
      {
         const double xi = xq[qx], eta = xq[qy];
         // bilinear geometry, vertices (0,0),(1,0),(0,1),(1,1)
         const double J00 = ax + eta * (bx - ax), J01 = cx + xi * (dx - cx);
         const double J10 = ay + eta * (by - ay), J11 = cy + xi * (dy - cy);
         const double det = J00 * J11 - J01 * J10;
         // J^-1 = adj / det with adj = [J11 -J01; -J10 J00]: the two 1/det and w |det| fold into w / |det|
         const double sc = wq[qx] * wq[qy] * fast_rcp(fabs(det));
         double *aq = a[3 * qy + qx];
         const double uxx = aq[0] * J11 - aq[1] * J10, uxy = aq[1] * J00 - aq[0] * J01;
         const double uyx = aq[2] * J11 - aq[3] * J10, uyy = aq[3] * J00 - aq[2] * J01;
         double sxx, syy, sxy;
         hooke_stress(lam, mu, sc, uxx, uyy, uxy + uyx, sxx, syy, sxy);
         aq[0] = J11 * sxx - J01 * sxy;
         aq[1] = J00 * sxy - J10 * sxx;
         aq[2] = J11 * sxy - J01 * syy;
         aq[3] = J00 * syy - J10 * sxy;
      }
   // transpose contractions
#pragma unroll
   for (int c = 0; c < 2; ++c)
   {
      double *y = c ? yy : yx;
      double t1[3][3], t0[3][3];  // [qx][j]
#pragma unroll
      for (int qx = 0; qx < 3; ++qx)
      {
         q2::interp_t(a[qx][2 * c], a[3 + qx][2 * c], a[6 + qx][2 * c], t1[qx]);
         t0[qx][0] = t0[qx][1] = t0[qx][2] = 0.;
         q2::deriv_t_add(a[qx][2 * c + 1], a[3 + qx][2 * c + 1], a[6 + qx][2 * c + 1], t0[qx]);
      }
#pragma unroll
      for (int j = 0; j < 3; ++j)
      {
         double v[3];
         q2::interp_t(t0[0][j], t0[1][j], t0[2][j], v);
         q2::deriv_t_add(t1[0][j], t1[1][j], t1[2][j], v);
         y[3 * j] = v[0], y[3 * j + 1] = v[1], y[3 * j + 2] = v[2];
      }
   }
}

__device__ __forceinline__ void red_add_f64(double *p, double v)
{
   asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

// byte offsets of the CTA's shared-memory buffers (from the host) and the bulk-copy sizes
struct PaLayout
{
   int li, cm;           // per-cell inputs of the current tile (one buffer)
   int nb, nb_bytes;     // 3 buffers of {tn, tp}: node ids and node -> refs offsets
   int tp;               // offset of tp inside one of them
   int tr, tr_bytes;     // trefs of the current tile
   int xs, xs_bytes;     // x values of the current tile
   int ye;               // element results
   int b_tn, b_tp;       // bytes copied per tile for tn / tp
};

struct PaArgs
{
   int64_t ncells;
   int ntiles;
   const int32_t *tnodes;
   const uint16_t *tptr, *trefs, *lidx;
   const double *geo;
   const uint32_t *cmask;
   const double *x;
   double *y;
   const double *flag;
   PaLayout L;
   int accumulate;  // y += A x (AddMultPA) instead of y = A x
};

__global__ void pa_zero_shared_kernel(int n, const int32_t *__restrict__ list, double *__restrict__ y,
                                      const double *__restrict__ flag)
{
   if (flag && *flag != 0.) return;
   const int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n) reinterpret_cast<double2 *>(y)[list[i]] = make_double2(0., 0.);
}

// Persistent CTAs, one thread per cell of a tile.  Thread 0 streams the tile plans and per-cell
// data (contiguous byte ranges) into shared memory with bulk copies one to two tiles ahead; the x
// values of tile i+1 are gathered with 16-byte cp.async (into the buffer tile i has just emptied into
// registers) while tile i is computed, so no thread waits on DRAM in steady state.  Per tile: inputs -> registers | element products -> ye |
// one thread per tile node sums its contributions and stores (interior) or reduces (tile boundary).
// 4 CTAs per SM (128 registers, no spills): compiled for 5 (96 registers, 136 bytes of spills) the Q2 apply is 9 %
// slower although the shared-memory footprint (45 KB) would allow it (profiles/r2_experiments.md)
template <int ET, bool DOT>
__global__ void __launch_bounds__(kPaThreads, 4) pa_tile_kernel(PaArgs A, ReduceScratch red, double *__restrict__ out)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, W = 2 * nv + 2, CT = kPaThreads, S = CT * nd;
   extern __shared__ __align__(128) unsigned char pa_sm[];
   __shared__ uint64_t fullG, fullN[3], fullT;
   if (A.flag && *A.flag != 0.) return;
   const int tid = threadIdx.x;
   const PaLayout &L = A.L;
   if (tid == 0)
   {
      mbar_init(&fullG, 1);
#pragma unroll
      for (int s = 0; s < 3; ++s) mbar_init(&fullN[s], 1);
      mbar_init(&fullT, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
   }
   __syncthreads();
   const int first = blockIdx.x, stride = gridDim.x;
   const int nmine = first < A.ntiles ? (A.ntiles - first + stride - 1) / stride : 0;
   const uint32_t b_cm = A.cmask ? CT * 4 : 0;
   auto tile_of = [&](int it) { return first + (int64_t)it * stride; };
   // thread 0 only
   auto load_N = [&](int it) {
      unsigned char *dst = pa_sm + L.nb + (size_t)(it % 3) * L.nb_bytes;
      const int64_t tile = tile_of(it);
      mbar_expect_tx(&fullN[it % 3], (uint32_t)(L.b_tn + L.b_tp));
      bulk_g2s(dst, A.tnodes + tile * S, (uint32_t)L.b_tn, &fullN[it % 3]);
      bulk_g2s(dst + L.tp, A.tptr + tile * (S + 8), (uint32_t)L.b_tp, &fullN[it % 3]);
   };
   auto load_T = [&](int it) {  // one buffer: reloaded after the scatter of the previous tile (barrier B2)
      mbar_expect_tx(&fullT, S * 2);
      bulk_g2s(pa_sm + L.tr, A.trefs + tile_of(it) * S, S * 2, &fullT);
   };
   auto load_G = [&](int it) {
      const int64_t tile = tile_of(it);
      mbar_expect_tx(&fullG, S * 2 + b_cm);
      bulk_g2s(pa_sm + L.li, A.lidx + tile * S, S * 2, &fullG);
      if (b_cm) bulk_g2s(pa_sm + L.cm, A.cmask + tile * CT, b_cm, &fullG);
   };
   const double2 *x2 = reinterpret_cast<const double2 *>(A.x);
   double2 *y2 = reinterpret_cast<double2 *>(A.y);
   double2 *ye = reinterpret_cast<double2 *>(pa_sm + L.ye);
   // gather the x values of tile it (its node list must have landed)
   auto gather_x = [&](int it) {
      const unsigned char *nb = pa_sm + L.nb + (size_t)(it % 3) * L.nb_bytes;
      const int nu = reinterpret_cast<const uint16_t *>(nb + L.tp)[0];
      const int32_t *tn = reinterpret_cast<const int32_t *>(nb);
      double2 *xs = reinterpret_cast<double2 *>(pa_sm + L.xs);
      for (int k = tid; k < nu; k += CT) cp_async16(xs + k, x2 + (tn[k] & 0x7fffffff));
   };
   double part = 0.;
   if (nmine > 0)
   {
      if (tid == 0)
      {
         load_N(0);
         if (nmine > 1) load_N(1);
         load_T(0);
         load_G(0);
      }
      mbar_wait(&fullN[0], 0);
      gather_x(0);
   }
   cp_async_commit();
   for (int it = 0; it < nmine; ++it)
   {
      // per-cell geometry + Lame pair straight from global memory (coalesced 16-byte loads, issued before the waits)
      double g[W];
      {
         const double2 *g2 = reinterpret_cast<const double2 *>(A.geo) + tile_of(it) * (W / 2) * CT + tid;
#pragma unroll
         for (int k = 0; k < W / 2; ++k)
         {
            const double2 v = ld_stream_d2(reinterpret_cast<const double *>(g2 + k * CT));
            g[2 * k] = v.x, g[2 * k + 1] = v.y;
         }
      }
      cp_async_wait<0>();
      __syncthreads();  // A: x of tile it visible; every thread is done with tile it - 1
      if (tid == 0 && it + 2 < nmine) load_N(it + 2);
      const int64_t e = tile_of(it) * CT + tid;
      const bool valid = e < A.ncells;
      const double2 *xs = reinterpret_cast<const double2 *>(pa_sm + L.xs);
      mbar_wait(&fullG, it & 1);
      uint32_t m = 0u;
      double ux[nd], uy[nd];
      {
         const uint16_t *lp = reinterpret_cast<const uint16_t *>(pa_sm + L.li) + tid;
         if (A.cmask) m = reinterpret_cast<const uint32_t *>(pa_sm + L.cm)[tid];
#pragma unroll
         for (int a = 0; a < nd; ++a)
         {
            const double2 v = xs[valid ? lp[a * CT] : 0];
            ux[a] = v.x, uy[a] = v.y;
         }
      }
      __syncthreads();  // B1: the per-cell inputs are in registers: the input buffers (G, xs) are free
      if (it + 1 < nmine)
      {
         if (tid == 0) load_G(it + 1);
         mbar_wait(&fullN[(it + 1) % 3], ((it + 1) / 3) & 1);
         gather_x(it + 1);
      }
      cp_async_commit();
      if (valid)
      {
         double yx[nd], yy[nd];
         if (m != 0u)
         {
#pragma unroll
            for (int a = 0; a < nd; ++a)
            {
               if ((m >> (2 * a)) & 1u) ux[a] = 0.;
               if ((m >> (2 * a + 1)) & 1u) uy[a] = 0.;
            }
         }
#if PA_EXP & 1
#pragma unroll
         for (int a = 0; a < nd; ++a) yx[a] = ux[a] * g[a % W], yy[a] = uy[a];
#else
         if (ET == FEMB200_Q2)
            local_apply_q2(g, ux, uy, yx, yy);
         else
            local_apply_tri<ET>(g, ux, uy, yx, yy);
#endif
         if (m != 0u)
         {
#pragma unroll
            for (int a = 0; a < nd; ++a)
            {
               if ((m >> (2 * a)) & 1u) yx[a] = 0.;
               if ((m >> (2 * a + 1)) & 1u) yy[a] = 0.;
            }
         }
         // contributions go to their node-sorted positions
         const uint16_t *pp = reinterpret_cast<const uint16_t *>(pa_sm + L.tr) + tid;
         mbar_wait(&fullT, it & 1);
#pragma unroll
         for (int a = 0; a < nd; ++a) ye[pp[a * CT]] = make_double2(yx[a], yy[a]);
      }
      __syncthreads();  // B2: ye complete, the scatter map of this tile is free
      if (tid == 0 && it + 1 < nmine) load_T(it + 1);
      // one thread per tile node: sum its (contiguous) contributions in a fixed order; KU nodes in flight
      const unsigned char *nb = pa_sm + L.nb + (size_t)(it % 3) * L.nb_bytes;
      const int32_t *tn = reinterpret_cast<const int32_t *>(nb);
      const uint16_t *tp = reinterpret_cast<const uint16_t *>(nb + L.tp);
      const int nu = (PA_EXP & 2) ? 0 : tp[0];
      constexpr int KU = ET == FEMB200_Q2 ? 5 : 3;
      for (int k0 = tid; k0 < nu; k0 += KU * CT)
      {
         int p0[KU], p1[KU];
         double2 acc[KU];
#pragma unroll
         for (int j = 0; j < KU; ++j)
         {
            const int k = k0 + j * CT;
            p0[j] = k < nu ? tp[1 + k] : 0;
            p1[j] = k < nu ? tp[2 + k] : 0;
            acc[j] = make_double2(0., 0.);
         }
         for (int r = 0;; ++r)
         {
            bool any = false;
#pragma unroll
            for (int j = 0; j < KU; ++j)
               if (p0[j] + r < p1[j])
               {
                  const double2 v = ye[p0[j] + r];
                  acc[j].x += v.x, acc[j].y += v.y;
                  any = true;
               }
            if (!any) break;
         }
#pragma unroll
         for (int j = 0; j < KU; ++j)
         {
            const int k = k0 + j * CT;
            if (k >= nu) continue;
            const int32_t id = tn[k];
            if (DOT)
            {  // <x, y> = sum over (tile, node) of x_node . partial: masked dofs contribute zeros
               const double2 xv = x2[id & 0x7fffffff];  // an L2 hit: gathered for this tile a moment ago
               part += xv.x * acc[j].x + xv.y * acc[j].y;
            }
            if (id < 0)
            {
               double *yp = A.y + 2 * (int64_t)(id & 0x7fffffff);
               red_add_f64(yp, acc[j].x);
               red_add_f64(yp + 1, acc[j].y);
            }
            else if (A.accumulate)
            {
               double2 o = y2[id];
               o.x += acc[j].x, o.y += acc[j].y;
               y2[id] = o;
            }
            else
               y2[id] = acc[j];
         }
      }
   }
   cp_async_wait<0>();
   if (DOT) block_reduce_finish<kPaThreads>(part, red, out);
}

// y[bc] = diag x[bc]; adds diag x[bc]^2 to the fused dot.  One CTA.
__global__ void __launch_bounds__(256)
pa_bc_fix_kernel(int nbc, const int32_t *__restrict__ list, double diag, const double *__restrict__ x,
                 double *__restrict__ y, const double *__restrict__ flag, double *__restrict__ out, bool accumulate)
{
   __shared__ double sh[8];
   if (flag && *flag != 0.) return;
   double part = 0.;
   for (int k = threadIdx.x; k < nbc; k += 256)
   {
      const int64_t i = list[k];
      const double xi = x[i];
      y[i] = accumulate ? y[i] + diag * xi : diag * xi;  // the element products left nothing on constrained dofs
      part += diag * xi * xi;
   }
   if (out)
   {
      const double t = block_sum<256>(part, sh);
      if (threadIdx.x == 0) *out += t;
   }
}

template <int ET>
__global__ void __launch_bounds__(kPaThreads)
pa_diag_kernel(int64_t ncells, const int32_t *__restrict__ cperm, const int32_t *__restrict__ dofmap,
               const double *__restrict__ geo, const uint32_t *__restrict__ cmask, double *__restrict__ diag)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq, W = 2 * nv + 2;
   const int64_t e = (int64_t)blockIdx.x * kPaThreads + threadIdx.x;
   if (e >= ncells) return;
   const double2 *g = reinterpret_cast<const double2 *>(geo) + (e / kPaThreads) * (W / 2) * kPaThreads + (e % kPaThreads);
   double xv[nv][2];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const double2 p = g[v * kPaThreads];
      xv[v][0] = p.x, xv[v][1] = p.y;
   }
   double D[9];
   const double2 lm = g[nv * kPaThreads];
   hooke_scaled(lm.x, lm.y, 1., D);
   double kd[nd][2];
#pragma unroll
   for (int a = 0; a < nd; ++a) kd[a][0] = kd[a][1] = 0.;
#pragma unroll 1
   for (int q = 0; q < nq; ++q)
   {
      double G[nd][2], phi[nv];
      const double w = qp_geometry<ET>(xv, q, G, phi);
#pragma unroll
      for (int a = 0; a < nd; ++a)
      {
         double k[4] = {0., 0., 0., 0.};
         bdb_block(G[a], G[a], D, w, k);
         kd[a][0] += k[0];
         kd[a][1] += k[3];
      }
   }
   const uint32_t m = cmask ? cmask[e] : 0u;
#pragma unroll
   for (int a = 0; a < nd; ++a)
   {
      double *dp = diag + 2 * (int64_t)dofmap[(int64_t)cperm[e] * nd + a];
      if (!((m >> (2 * a)) & 1u)) red_add_f64(dp, kd[a][0]);
      if (!((m >> (2 * a + 1)) & 1u)) red_add_f64(dp + 1, kd[a][1]);
   }
}

__global__ void pa_diag_bc_kernel(int nbc, const int32_t *__restrict__ list, double diag, double *__restrict__ d)
{
   const int k = blockIdx.x * blockDim.x + threadIdx.x;
   if (k < nbc) d[list[k]] = diag;
}

// ---- multigrid: the first coarse operator of a p-coarsening (P2 -> P1, Q2 -> Q1 on the same cells) ----------------
// Restricted to a cell, the global prolongation is the fixed element interpolation P_e (fine local dof a, coarse local
// vertex v): P2 -> P1 is 1 at the vertices and 1/2, 1/2 at the midpoint of an edge (edge 3 + i is opposite vertex i);
// Q2 -> Q1 is the tensor product of the 1-D rows (1, 0), (1/2, 1/2), (0, 1), coarse order (v00, v10, v01, v11) = cx + 2 cy.
// So P^T A P = sum_e P_e^T K_e P_e, with the rows of the constrained fine dofs of P_e zeroed (cmask).
template <int ET>
__device__ __forceinline__ double pcoarse_weight(int a, int v)
{
   if constexpr (ET == FEMB200_Q2)
   {
      const int ix = a % 3, iy = a / 3, cx = v & 1, cy = v >> 1;
      const double wx = ix == 1 ? 0.5 : (ix == 2 * cx ? 1. : 0.), wy = iy == 1 ? 0.5 : (iy == 2 * cy ? 1. : 0.);
      return wx * wy;
   }
   else
      return a < 3 ? (a == v ? 1. : 0.) : (a - 3 == v ? 0. : 0.5);
}

// kc[cell] = P_e^T K_e P_e, (2 nv) x (2 nv) row-major over the interleaved coarse dofs (2 v + c), one thread per cell (tile
// order), the PA quadrature and geometry; fixed summation order (deterministic)
template <int ET>
__global__ void __launch_bounds__(kPaThreads)
pa_galerkin_kernel(int64_t ncells, const int32_t *__restrict__ cperm, const double *__restrict__ geo,
                   const uint32_t *__restrict__ cmask, double *__restrict__ kc)
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq, W = 2 * nv + 2, N2 = 2 * nv;
   const int64_t e = (int64_t)blockIdx.x * kPaThreads + threadIdx.x;
   if (e >= ncells) return;
   const double2 *g = reinterpret_cast<const double2 *>(geo) + (e / kPaThreads) * (W / 2) * kPaThreads + (e % kPaThreads);
   double xv[nv][2];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const double2 p = g[v * kPaThreads];
      xv[v][0] = p.x, xv[v][1] = p.y;
   }
   double D[9];
   const double2 lm = g[nv * kPaThreads];
   hooke_scaled(lm.x, lm.y, 1., D);
   const uint32_t m = cmask ? cmask[e] : 0u;
   double K[N2][N2];
#pragma unroll
   for (int i = 0; i < N2; ++i)
#pragma unroll
      for (int j = 0; j < N2; ++j) K[i][j] = 0.;
#pragma unroll 1
   for (int q = 0; q < nq; ++q)
   {
      double G[nd][2], phi[nv];
      const double w = qp_geometry<ET>(xv, q, G, phi);
      // gradient of coarse basis function v as seen by displacement component c: sum_a P_e[a][v] G_a over the free (a, c)
      double gc[2][nv][2];
#pragma unroll
      for (int c = 0; c < 2; ++c)
#pragma unroll
         for (int v = 0; v < nv; ++v) gc[c][v][0] = gc[c][v][1] = 0.;
#pragma unroll
      for (int a = 0; a < nd; ++a)
#pragma unroll
         for (int v = 0; v < nv; ++v)
         {
            const double p = pcoarse_weight<ET>(a, v);
            if (p == 0.) continue;
#pragma unroll
            for (int c = 0; c < 2; ++c)
               if (!((m >> (2 * a + c)) & 1u)) gc[c][v][0] += p * G[a][0], gc[c][v][1] += p * G[a][1];
         }
      // K[2v + c][2u + d] += w B_c(gc[c][v])^T D B_d(gc[d][u]), B_x(g) = (g0, 0, g1), B_y(g) = (0, g1, g0) (bdb_block)
#pragma unroll
      for (int v = 0; v < nv; ++v)
#pragma unroll
         for (int c = 0; c < 2; ++c)
         {
            const double *h = gc[c][v];
            double r[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) r[k] = c == 0 ? h[0] * D[k] + h[1] * D[6 + k] : h[1] * D[3 + k] + h[0] * D[6 + k];
#pragma unroll
            for (int u = 0; u < nv; ++u)
#pragma unroll
               for (int d = 0; d < 2; ++d)
               {
                  const double *f = gc[d][u];
                  const double s = d == 0 ? r[0] * f[0] + r[2] * f[1] : r[1] * f[1] + r[2] * f[0];
                  K[2 * v + c][2 * u + d] += w * s;
               }
         }
   }
   double *out = kc + (int64_t)cperm[e] * (N2 * N2);
#pragma unroll
   for (int i = 0; i < N2; ++i)
#pragma unroll
      for (int j = 0; j < N2; j += 2) *reinterpret_cast<double2 *>(out + i * N2 + j) = make_double2(K[i][j], K[i][j + 1]);
}

// Coarse CSR values from the per-cell matrices through the coarse plan's visit records (plan.cuh): one thread per node
// row (the plan's tile order), its visits in the plan's order; the first visit to reach a slot stores, later ones add.
// One writer per row, no atomics: deterministic.  Triangles (P1) keep the columns of a record in rotated order.
__global__ void __launch_bounds__(kAsmR)
pa_galerkin_gather_kernel(int64_t nnodes, int nc, bool rotated, const int32_t *__restrict__ nptr,
                          const VisitRec *__restrict__ vrec, const uint8_t *__restrict__ perm,
                          const uint16_t *__restrict__ voff, const int64_t *__restrict__ brp, const double *__restrict__ kc,
                          double *__restrict__ values)
{
   const int rank = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR;
   if (rank >= (int)min((int64_t)kAsmR, nnodes - n0)) return;
   const int64_t I = n0 + perm[n0 + rank];
   const int cnt = nptr[I + 1] - nptr[I];
   const uint16_t *vo = voff + (int64_t)blockIdx.x * kAsmLevels;
   const uint4 *rec = reinterpret_cast<const uint4 *>(vrec + nptr[n0]) + rank;
   const int64_t b0 = brp[I];
   const int deg = (int)(brp[I + 1] - b0);
   double *row0 = values + 4 * b0, *row1 = row0 + 2 * deg;
   const int n2 = 2 * nc;
   for (int j = 0; j < cnt; ++j)
   {
      const Visit r(rec[vo[j]]);
      const double *k0 = kc + (int64_t)r.e * n2 * n2 + (int64_t)(2 * r.a) * n2, *k1 = k0 + n2;
      for (int b = 0; b < nc; ++b)
      {
         const int t = rotated ? (b - (int)r.a + 3) % 3 : b;
         const int s = r.slot(t);
         const double2 v0 = *reinterpret_cast<const double2 *>(k0 + 2 * b), v1 = *reinterpret_cast<const double2 *>(k1 + 2 * b);
         double2 *o0 = reinterpret_cast<double2 *>(row0 + 2 * s), *o1 = reinterpret_cast<double2 *>(row1 + 2 * s);
         if (r.is_first(t))
            *o0 = v0, *o1 = v1;
         else
         {
            const double2 a0 = *o0, a1 = *o1;
            *o0 = make_double2(a0.x + v0.x, a0.y + v0.y), *o1 = make_double2(a1.x + v1.x, a1.y + v1.y);
         }
      }
   }
}

// coarse vertices v with a non-zero P_e[a][v] (bit v) of the element interpolation (pcoarse_weight): Q2 -> Q1 (nd = 9)
// or P2 -> P1 (nd = 6)
__device__ __forceinline__ unsigned pcoarse_support(int nd, int a)
{
   if (nd == 9)
   {
      const int ix = a % 3, iy = a / 3;
      const unsigned mx = ix == 0 ? 1u : (ix == 2 ? 2u : 3u), my = iy == 0 ? 1u : (iy == 2 ? 2u : 3u);
      unsigned sup = 0u;
      for (int v = 0; v < 4; ++v)
         if (((mx >> (v & 1)) & 1u) && ((my >> (v >> 1)) & 1u)) sup |= 1u << v;
      return sup;
   }
   return a < 3 ? 1u << a : 7u & ~(1u << (a - 3));
}

// err = 1 unless, for every fine cell e and local dof a, the transfer map row of the dof names exactly the coarse nodes
// of coarse cell e that P_e gives it a weight on: its coincident vertex, the two ends of its edge, the four vertices of
// its quad (the element Galerkin step uses P_e; restriction and prolongation use the map: they must agree)
__global__ void pa_pcoarse_check_kernel(int64_t ncells, int nd, int nc, const int32_t *__restrict__ fdofmap,
                                        const int32_t *__restrict__ cdofmap, const int32_t *__restrict__ map, int width,
                                        int *__restrict__ err)
{
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   int32_t cv[4];
   for (int v = 0; v < nc; ++v) cv[v] = cdofmap[e * nc + v];
   for (int a = 0; a < nd; ++a)
   {
      const unsigned sup = pcoarse_support(nd, a);
      const int32_t *row = map + (int64_t)fdofmap[e * nd + a] * width;
      bool ok = true;
      for (int k = 0; k < width; ++k)
      {  // every entry is a supporting coarse vertex
         bool in = false;
         for (int v = 0; v < nc; ++v) in = in || (((sup >> v) & 1u) && row[k] == cv[v]);
         ok = ok && in;
      }
      for (int v = 0; v < nc; ++v)
         if ((sup >> v) & 1u)
         {  // every supporting coarse vertex is an entry
            bool in = false;
            for (int k = 0; k < width; ++k) in = in || row[k] == cv[v];
            ok = ok && in;
         }
      if (!ok) *err = 1;
   }
}

static PaLayout pa_layout(const femb200_pa *pa)
{
   const int CT = kPaThreads, S = CT * pa->nd;
   auto up = [](int v) { return (v + 127) & ~127; };
   PaLayout L;
   int o = 0;
   L.li = o, o += up(S * 2);
   L.cm = o, o += up(CT * 4);
   L.b_tn = ((pa->max_uniq + 3) & ~3) * 4;
   L.b_tp = ((pa->max_uniq + 2 + 7) & ~7) * 2;
   L.tp = up(L.b_tn);
   L.nb_bytes = L.tp + up(L.b_tp);
   L.nb = o, o += 3 * L.nb_bytes;
   L.tr_bytes = up(S * 2);
   L.tr = o, o += L.tr_bytes;
   L.xs_bytes = up(pa->max_uniq * 16);
   L.xs = o, o += L.xs_bytes;
   L.ye = o;
   return L;
}

template <int ET>
static int pa_apply_t(const femb200_pa *pa, const double *d_x, double *d_y, const double *d_flag, double *d_dot_out,
                      cudaStream_t st, bool accumulate)
{
   const PaLayout L = pa_layout(pa);
   const size_t smem = (size_t)L.ye + sizeof(double2) * (size_t)kPaThreads * Elem<ET>::nd;
   const size_t lim = devinfo().smem_optin - 1024;
   FEMB_CHECK(smem <= lim, "pa_apply: tile needs %zu bytes of shared memory", smem);
   static bool attr_done = false;
   if (!attr_done)
   {
      FEMB_CUDA(cudaFuncSetAttribute(pa_tile_kernel<ET, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lim));
      FEMB_CUDA(cudaFuncSetAttribute(pa_tile_kernel<ET, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lim));
      attr_done = true;
   }
   int per_sm = 1;
   if (d_dot_out)
      FEMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pa_tile_kernel<ET, true>, kPaThreads, smem));
   else
      FEMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pa_tile_kernel<ET, false>, kPaThreads, smem));
   const unsigned grid = (unsigned)std::min<int64_t>(pa->ntiles, (int64_t)devinfo().sm_count * std::max(1, per_sm));
   PaArgs A{pa->ncells, (int)pa->ntiles, pa->tnodes, pa->tptr, pa->trefs, pa->lidx, pa->geo, pa->cmask, d_x, d_y, d_flag, L,
            accumulate ? 1 : 0};
   if (d_dot_out)
   {
      ReduceScratch red;
      if (int rc = reduce_scratch(grid, st, &red)) return rc;
      pa_tile_kernel<ET, true><<<grid, kPaThreads, smem, st>>>(A, red, d_dot_out);
   }
   else
      pa_tile_kernel<ET, false><<<grid, kPaThreads, smem, st>>>(A, ReduceScratch{nullptr, nullptr}, nullptr);
   FEMB_LAUNCH_CHECK();
   return 0;
}

int pa_apply_launch(const femb200_pa *pa, const double *d_x, double *d_y, const double *d_flag, double *d_dot_out,
                    cudaStream_t st, bool accumulate)
{
   // only the nodes shared between tiles are accumulated with reductions: zero those (y = A x); with
   // accumulate (y += A x) the reductions add to what y holds and interior nodes read-modify-write
   if (pa->nshared > 0 && !accumulate)
   {
      pa_zero_shared_kernel<<<(unsigned)cdiv(pa->nshared, 256), 256, 0, st>>>(pa->nshared, pa->shared_nodes, d_y, d_flag);
      FEMB_LAUNCH_CHECK();
   }
   int rc;
   switch (pa->etype)
   {
      case FEMB200_P1: rc = pa_apply_t<FEMB200_P1>(pa, d_x, d_y, d_flag, d_dot_out, st, accumulate); break;
      case FEMB200_P2: rc = pa_apply_t<FEMB200_P2>(pa, d_x, d_y, d_flag, d_dot_out, st, accumulate); break;
      default: rc = pa_apply_t<FEMB200_Q2>(pa, d_x, d_y, d_flag, d_dot_out, st, accumulate);
   }
   if (rc) return rc;
   if (pa->nbc > 0)
   {
      pa_bc_fix_kernel<<<1, 256, 0, st>>>(pa->nbc, pa->bc_dofs, pa->diag, d_x, d_y, d_flag, d_dot_out, accumulate);
      FEMB_LAUNCH_CHECK();
   }
   return 0;
}

// ---- setup driver -------------------------------------------------------------------
template <typename T>
static int pa_alloc(femb200_pa *pa, T **p, size_t n)
{
   const size_t b = sizeof(T) * (n ? n : 1);
   if (cudaMalloc(p, b) != cudaSuccess) return set_error("pa_create: cudaMalloc of %zu bytes failed", b);
   pa->bytes += b;
   return 0;
}

template <int ND>
static void pa_tile_build(femb200_pa *pa, int end_bit, int32_t *ntouch, cudaStream_t st)
{
   pa_tile_build_kernel<ND, kPaThreads><<<(unsigned)pa->ntiles, kPaThreads, 0, st>>>(
      pa->ncells, pa->nnodes, end_bit, pa->dofmap, pa->cperm, pa->tnodes, pa->tptr, pa->trefs, pa->lidx, pa->tcount,
      ntouch);
}

static int pa_build_tiles(femb200_pa *pa, const int32_t *d_xdofmap, const double *d_x, int xs, cudaStream_t st)
{
   const int64_t nc = pa->ncells;
   const int CT = kPaThreads, S = CT * pa->nd;
   pa->ct = CT;
   pa->ntiles = cdiv(nc, CT);
   // 1. Morton order of the cell centroids
   float *cx = nullptr, *cy = nullptr, *bb = nullptr;
   uint32_t *key = nullptr, *key2 = nullptr;
   int32_t *id = nullptr, *ntouch = nullptr, *count = nullptr;
   void *tmp = nullptr;
   auto cleanup = [&](int rc) {
      cudaFree(cx), cudaFree(cy), cudaFree(bb), cudaFree(key), cudaFree(key2), cudaFree(id), cudaFree(ntouch);
      cudaFree(count), cudaFree(tmp);
      return rc;
   };
   size_t scratch = 0;
   femb200_pa dummy;  // setup scratch is not counted in pa->bytes
   if (pa_alloc(&dummy, &cx, (size_t)nc) || pa_alloc(&dummy, &cy, (size_t)nc) || pa_alloc(&dummy, &bb, 4) ||
       pa_alloc(&dummy, &key, (size_t)nc) || pa_alloc(&dummy, &key2, (size_t)nc) || pa_alloc(&dummy, &id, (size_t)nc) ||
       pa_alloc(&dummy, &ntouch, (size_t)pa->nnodes) || pa_alloc(&dummy, &count, 1) || pa_alloc(pa, &pa->cperm, (size_t)nc))
      return cleanup(1);
   const unsigned gc = (unsigned)cdiv(nc, 256);
   pa_centroid_kernel<<<gc, 256, 0, st>>>(nc, pa->nv, d_xdofmap, d_x, xs, cx, cy);
   size_t need = 0, n1 = 0;
   cub::DeviceReduce::Min(nullptr, need, cx, bb, (int)nc, st);
   cub::DeviceRadixSort::SortPairs(nullptr, n1, key, key2, id, pa->cperm, (int)nc, 0, 32, st);
   scratch = std::max(need, n1);
   if (cudaMalloc(&tmp, scratch) != cudaSuccess) return cleanup(set_error("pa_create: cudaMalloc of %zu bytes failed", scratch));
   cub::DeviceReduce::Min(tmp, scratch, cx, bb + 0, (int)nc, st);
   cub::DeviceReduce::Max(tmp, scratch, cx, bb + 1, (int)nc, st);
   cub::DeviceReduce::Min(tmp, scratch, cy, bb + 2, (int)nc, st);
   cub::DeviceReduce::Max(tmp, scratch, cy, bb + 3, (int)nc, st);
   pa_morton_kernel<<<gc, 256, 0, st>>>(nc, cx, cy, bb, key, id);
   cub::DeviceRadixSort::SortPairs(tmp, scratch, key, key2, id, pa->cperm, (int)nc, 0, 32, st);
   // 2. per-tile node lists
   const size_t nt = (size_t)pa->ntiles;
   if (pa_alloc(pa, &pa->tcount, nt) || pa_alloc(pa, &pa->tnodes, nt * S) || pa_alloc(pa, &pa->tptr, nt * (S + 8)) ||
       pa_alloc(pa, &pa->trefs, nt * S) || pa_alloc(pa, &pa->lidx, nt * S))
      return cleanup(1);
   cudaMemsetAsync(ntouch, 0, sizeof(int32_t) * (size_t)pa->nnodes, st);
   int end_bit = 1;
   while (end_bit < 32 && (pa->nnodes >> end_bit) != 0) ++end_bit;
   switch (pa->nd)
   {
      case 3: pa_tile_build<3>(pa, end_bit, ntouch, st); break;
      case 6: pa_tile_build<6>(pa, end_bit, ntouch, st); break;
      default: pa_tile_build<9>(pa, end_bit, ntouch, st);
   }
   pa_tile_flag_kernel<<<(unsigned)pa->ntiles, 128, 0, st>>>(pa->ntiles, S, pa->tcount, ntouch, pa->tnodes);
   // 3. nodes shared between tiles, largest tile
   int32_t *mx = count;
   cub::DeviceReduce::Max(tmp, scratch, pa->tcount, mx, (int)pa->ntiles, st);
   int32_t h = 0;
   cudaMemcpyAsync(&h, mx, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
   if (cudaStreamSynchronize(st) != cudaSuccess)
      return cleanup(set_error("pa_create: tile build failed: %s", cudaGetErrorString(cudaGetLastError())));
   pa->max_uniq = h;
   cudaMemsetAsync(count, 0, sizeof(int32_t), st);
   const unsigned gn = (unsigned)cdiv(pa->nnodes, 256);
   pa_shared_list_kernel<<<gn, 256, 0, st>>>(pa->nnodes, ntouch, nullptr, count);
   cudaMemcpyAsync(&h, count, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
   if (cudaStreamSynchronize(st) != cudaSuccess)
      return cleanup(set_error("pa_create: shared-node count failed: %s", cudaGetErrorString(cudaGetLastError())));
   pa->nshared = h;
   if (pa_alloc(pa, &pa->shared_nodes, (size_t)h)) return cleanup(1);
   cudaMemsetAsync(count, 0, sizeof(int32_t), st);
   pa_shared_list_kernel<<<gn, 256, 0, st>>>(pa->nnodes, ntouch, pa->shared_nodes, count);
   if (cudaStreamSynchronize(st) != cudaSuccess)
      return cleanup(set_error("pa_create: shared-node list failed: %s", cudaGetErrorString(cudaGetLastError())));
   return cleanup(0);
}

}  // namespace femb

using namespace femb;

extern "C" void femb200_pa_destroy(femb200_pa *pa)
{
   if (!pa) return;
   cudaFree(pa->cperm);
   cudaFree(pa->geo);
   cudaFree(pa->tcount);
   cudaFree(pa->tnodes);
   cudaFree(pa->tptr);
   cudaFree(pa->trefs);
   cudaFree(pa->lidx);
   cudaFree(pa->shared_nodes);
   cudaFree(pa->cmask);
   cudaFree(pa->bc);
   cudaFree(pa->bc_dofs);
   delete pa;
}

extern "C" int femb200_pa_create(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap,
                                 const int32_t *d_xdofmap, const double *d_x, int x_stride, const double *d_E, double nu,
                                 void *stream, femb200_pa **out)
{
   FEMB_CHECK(out != nullptr, "pa_create: out is null");
   *out = nullptr;
   FEMB_REFUSE_Q1(etype, "pa_create");
   FEMB_CHECK(etype >= FEMB200_P1 && etype <= FEMB200_Q2, "pa_create: unknown element family %d", etype);
   FEMB_CHECK(nnodes > 0 && ncells > 0, "pa_create: empty mesh");
   FEMB_CHECK(d_dofmap && d_xdofmap && d_x && d_E, "pa_create: null argument");
   FEMB_CHECK(x_stride == 2 || x_stride == 3, "pa_create: x_stride must be 2 or 3, got %d", x_stride);
   FEMB_CHECK(ncells < (int64_t)1 << 31 && nnodes < (int64_t)1 << 31, "pa_create: mesh too large for 32-bit local indices");
   femb200_pa *pa = new femb200_pa();
   pa->etype = etype, pa->nd = elem_nd(etype), pa->nv = elem_nv(etype);
   pa->nnodes = nnodes, pa->ncells = ncells, pa->dofmap = d_dofmap;
   cudaStream_t st = as_stream(stream);
   if (pa_build_tiles(pa, d_xdofmap, d_x, x_stride, st))
   {
      femb200_pa_destroy(pa);
      return 1;
   }
   const size_t W = 2 * (size_t)pa->nv + 2;
   const size_t padded = (size_t)pa->ntiles * kPaThreads;
   if (pa_alloc(pa, &pa->geo, W * padded) || cudaMemsetAsync(pa->geo, 0, sizeof(double) * W * padded, st) != cudaSuccess)
   {
      femb200_pa_destroy(pa);
      return 1;
   }
   const LameCoef lc = lame_coef(nu);
   const unsigned grid = (unsigned)cdiv(ncells, 256);
   if (etype == FEMB200_Q2)
      pa_setup_kernel<FEMB200_Q2><<<grid, 256, 0, st>>>(ncells, pa->cperm, d_xdofmap, d_x, x_stride, d_E, lc, pa->geo);
   else
      pa_setup_kernel<FEMB200_P1><<<grid, 256, 0, st>>>(ncells, pa->cperm, d_xdofmap, d_x, x_stride, d_E, lc, pa->geo);
   if (cudaGetLastError() != cudaSuccess)
   {
      femb200_pa_destroy(pa);
      return set_error("pa_create: setup launch failed");
   }
   *out = pa;
   return 0;
}

extern "C" int femb200_pa_set_dirichlet(femb200_pa *pa, const uint8_t *d_bc, double diag, void *stream)
{
   FEMB_CHECK(pa != nullptr, "pa_set_dirichlet: null operator");
   cudaStream_t st = as_stream(stream);
   cudaFree(pa->cmask), cudaFree(pa->bc), cudaFree(pa->bc_dofs);
   pa->cmask = nullptr, pa->bc = nullptr, pa->bc_dofs = nullptr, pa->nbc = 0;
   pa->diag = diag;
   if (!d_bc) return 0;
   const int64_t nd = 2 * pa->nnodes;
   int32_t *count = nullptr;
   // every failure below leaves the operator unconstrained and owns nothing
   auto fail = [&](const char *what) {
      cudaFree(count);
      cudaFree(pa->cmask), cudaFree(pa->bc), cudaFree(pa->bc_dofs);
      pa->cmask = nullptr, pa->bc = nullptr, pa->bc_dofs = nullptr, pa->nbc = 0;
      return set_error("pa_set_dirichlet: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
   };
   if (cudaMalloc(&pa->bc, (size_t)nd) != cudaSuccess ||
       cudaMalloc(&pa->cmask, sizeof(uint32_t) * (size_t)pa->ntiles * kPaThreads) != cudaSuccess ||
       cudaMalloc(&count, sizeof(int32_t)) != cudaSuccess)
      return fail("cudaMalloc");
   if (cudaMemsetAsync(pa->cmask, 0, sizeof(uint32_t) * (size_t)pa->ntiles * kPaThreads, st) != cudaSuccess ||
       cudaMemcpyAsync(pa->bc, d_bc, (size_t)nd, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
       cudaMemsetAsync(count, 0, sizeof(int32_t), st) != cudaSuccess)
      return fail("copy");
   pa_cmask_kernel<<<(unsigned)cdiv(pa->ncells, 256), 256, 0, st>>>(pa->ncells, pa->nd, pa->cperm, pa->dofmap, pa->bc,
                                                                    pa->cmask);
   pa_bc_list_kernel<<<(unsigned)cdiv(nd, 256), 256, 0, st>>>(nd, pa->bc, nullptr, count);
   int32_t n = 0;
   cudaMemcpyAsync(&n, count, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
   if (cudaStreamSynchronize(st) != cudaSuccess) return fail("constrained-dof count");
   if (cudaMalloc(&pa->bc_dofs, sizeof(int32_t) * (size_t)(n ? n : 1)) != cudaSuccess) return fail("cudaMalloc");
   cudaMemsetAsync(count, 0, sizeof(int32_t), st);
   pa_bc_list_kernel<<<(unsigned)cdiv(nd, 256), 256, 0, st>>>(nd, pa->bc, pa->bc_dofs, count);
   cudaStreamSynchronize(st);
   cudaFree(count);
   pa->nbc = n;
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_pa_apply(const femb200_pa *pa, const double *d_x, double *d_y, void *stream)
{
   FEMB_CHECK(pa && d_x && d_y, "pa_apply: null argument");
   FEMB_CHECK(d_x != d_y, "pa_apply: x and y must not alias");
   return pa_apply_launch(pa, d_x, d_y, nullptr, nullptr, as_stream(stream), false);
}

int64_t pa_num_dofs(const femb200_pa *pa) { return pa ? 2 * pa->nnodes : 0; }
// BilinearFormIntegrator::AddMultPA(x, y): y += A x, accumulated in the node phase of the apply kernel (no scratch
// vector, no extra pass); d_work is unused and may be NULL (kept for the round-1 signature)
extern "C" int femb200_add_mult_pa(const femb200_pa *pa, int64_t ndofs, const double *d_x, double *d_y, double *d_work,
                                   void *stream)
{
   (void)d_work;
   FEMB_CHECK(pa && d_x && d_y, "add_mult_pa: null argument");
   FEMB_CHECK(d_x != d_y, "add_mult_pa: x and y must not alias");
   FEMB_CHECK(ndofs == 2 * pa->nnodes, "add_mult_pa: ndofs = %lld, the operator has %lld", (long long)ndofs,
              (long long)(2 * pa->nnodes));
   return pa_apply_launch(pa, d_x, d_y, nullptr, nullptr, as_stream(stream), true);
}

extern "C" int femb200_pa_diagonal(const femb200_pa *pa, double *d_diag, void *stream)
{
   FEMB_CHECK(pa && d_diag, "pa_diagonal: null argument");
   cudaStream_t st = as_stream(stream);
   FEMB_CUDA(cudaMemsetAsync(d_diag, 0, sizeof(double) * 2 * (size_t)pa->nnodes, st));
   const unsigned grid = (unsigned)cdiv(pa->ncells, kPaThreads);
   switch (pa->etype)
   {
      case FEMB200_P1:
         pa_diag_kernel<FEMB200_P1><<<grid, kPaThreads, 0, st>>>(pa->ncells, pa->cperm, pa->dofmap, pa->geo, pa->cmask, d_diag);
         break;
      case FEMB200_P2:
         pa_diag_kernel<FEMB200_P2><<<grid, kPaThreads, 0, st>>>(pa->ncells, pa->cperm, pa->dofmap, pa->geo, pa->cmask, d_diag);
         break;
      default:
         pa_diag_kernel<FEMB200_Q2><<<grid, kPaThreads, 0, st>>>(pa->ncells, pa->cperm, pa->dofmap, pa->geo, pa->cmask, d_diag);
   }
   FEMB_LAUNCH_CHECK();
   if (pa->nbc > 0)
   {
      pa_diag_bc_kernel<<<(unsigned)cdiv(pa->nbc, 256), 256, 0, st>>>(pa->nbc, pa->bc_dofs, pa->diag, d_diag);
      FEMB_LAUNCH_CHECK();
   }
   return 0;
}

// ---- internal interface of the multigrid handle (mg.cu): the operator stays private ------------------------------
namespace femb {

int pa_mg_info(const femb200_pa *pa, int *etype, int64_t *nnodes, int64_t *ncells)
{
   FEMB_CHECK(pa, "mg_create: null matrix-free operator");
   *etype = pa->etype, *nnodes = pa->nnodes, *ncells = pa->ncells;
   return 0;
}

// the operator's current Dirichlet marker (femb200_pa_set_dirichlet replaces it), or null
const uint8_t *pa_dirichlet_marker(const femb200_pa *pa) { return pa->bc; }

static int pa_coarse_family(const femb200_pa *pa, const femb200_plan *coarse, const char *who)
{
   const int want = pa->etype == FEMB200_Q2 ? FEMB200_Q1 : FEMB200_P1;
   FEMB_CHECK(pa->etype != FEMB200_P1 && coarse->etype == want && coarse->ncells == pa->ncells,
              "%s: the first coarse level of a matrix-free operator must be a p-coarsening (P2 -> P1 or Q2 -> Q1 on the same "
              "cells, in the same order)", who);
   return 0;
}

int pa_check_pcoarsening(const femb200_pa *pa, const femb200_plan *coarse, const int32_t *d_map, int width, int *d_err,
                         cudaStream_t st)
{
   if (int rc = pa_coarse_family(pa, coarse, "mg_create")) return rc;
   FEMB_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), st));
   pa_pcoarse_check_kernel<<<(unsigned)cdiv(pa->ncells, 256), 256, 0, st>>>(pa->ncells, pa->nd, coarse->nd, pa->dofmap,
                                                                             coarse->dofmap, d_map, width, d_err);
   FEMB_LAUNCH_CHECK();
   int herr = 0;
   FEMB_CUDA(cudaMemcpyAsync(&herr, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
   FEMB_CUDA(cudaStreamSynchronize(st));
   FEMB_CHECK(herr == 0,
              "mg_create: the first coarse level of a matrix-free operator must be a p-coarsening (P2 -> P1 or Q2 -> Q1 on "
              "the same cells, in the same order): the transfer map of a fine cell's nodes is not the element interpolation "
              "from the coarse cell with the same number (vertices coincident, edge midpoints and centres from its vertices)");
   return 0;
}

// coarse values = P^T A P for the p-coarsening onto `coarse` (Dirichlet rows / columns of the coarse plan not applied).
// The per-cell scratch ((2 nv)^2 doubles per cell: 8.6 GB for 16.8 M Q2 cells) lives for the call only, stream-ordered.
int pa_element_galerkin(const femb200_pa *pa, const femb200_plan *coarse, double *d_values, cudaStream_t st)
{
   if (int rc = pa_coarse_family(pa, coarse, "mg_galerkin")) return rc;
   const unsigned grid = (unsigned)cdiv(pa->ncells, kPaThreads);
   double *d_kc = nullptr;
   FEMB_CUDA(cudaMallocAsync(&d_kc, sizeof(double) * (size_t)pa->ncells * (size_t)(4 * pa->nv * pa->nv), st));
   if (pa->etype == FEMB200_Q2)
      pa_galerkin_kernel<FEMB200_Q2><<<grid, kPaThreads, 0, st>>>(pa->ncells, pa->cperm, pa->geo, pa->cmask, d_kc);
   else
      pa_galerkin_kernel<FEMB200_P2><<<grid, kPaThreads, 0, st>>>(pa->ncells, pa->cperm, pa->geo, pa->cmask, d_kc);
   pa_galerkin_gather_kernel<<<(unsigned)cdiv(coarse->nnodes, kAsmR), kAsmR, 0, st>>>(
       coarse->nnodes, coarse->nd, elem_is_triangle(coarse->etype), coarse->nptr, coarse->vrec, coarse->perm, coarse->voff,
       coarse->brp, d_kc, d_values);
   const cudaError_t e = cudaGetLastError();
   FEMB_CUDA(cudaFreeAsync(d_kc, st));
   FEMB_CHECK(e == cudaSuccess, "mg_galerkin: element Galerkin launch failed: %s", cudaGetErrorString(e));
   return 0;
}

}  // namespace femb
