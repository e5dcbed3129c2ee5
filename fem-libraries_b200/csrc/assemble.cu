// assemble.cu -- write-once gather assembly of the global tangent matrix.
//
// Role in the reference: the setJ lambda (F.cc:847-862) = MatZeroEntries +
// dolfinx assemble_matrix(set_block_fn(A, ADD_VALUES), J, bcs) + set_diagonal +
// MatAssembly, i.e. per cell: tabulate_tensor -> zero Dirichlet rows/cols ->
// MatSetValuesBlockedLocal (binary searches, read-modify-write of the CSR); on the
// MFEM side ParNonlinearForm::GetGradient -> AssembleElementGrad (M.cc:639-916) ->
// SparseMatrix::AddSubMatrix.
//
// B200 design: no scatter, no atomics, no zero-fill.  One thread owns one block
// row (node I) of the matrix.  It walks the cells incident to I (VisitRec list of
// the plan), computes only the 2 x 2nd row slice of each element matrix that
// belongs to I, and accumulates it into a shared-memory image of its CSR rows
// (first contribution stores, later ones add: the plan pre-computes which is
// which).  A CTA owns R consecutive nodes, whose CSR values are one contiguous
// byte range: after the tile is complete it is streamed out with 16-byte coalesced
// stores, every value written exactly once.  HBM traffic = nnz*8 B written +
// ~120 B/cell of maps and geometry read (DESIGN.md, kernel K1+K3).
//
// Fast path (P1/P2, d = 0): on a straight-sided triangle with constant D the P2
// element matrix is an exact linear combination of the nine 2x2 blocks
//   W^{cd} = |T| g_c^t C g_d ,  g_c = grad lambda_c   (c,d = vertices)
// (these are the P1 stiffness blocks, M.cc:699-704,885-887 with w = |T|):
//   vertex a / vertex b :  W^{aa}  or  -W^{ab}/3
//   vertex p / edge (p,q):  4/3 W^{pq};  vertex / opposite edge: 0
//   edge (p,q) / edge (r,s): 4/3 [(1+d_qs) W^{pr} + (1+d_qr) W^{ps} + (1+d_ps) W^{qr} + (1+d_pr) W^{qs}]
// which is what the 3-point rule integrates exactly (SURVEY.md A.9, 8c).  The row
// owner relabels the triangle so that its own local index is vertex 0 / edge 0:
// only 3 W blocks are needed per visit.
//
// Kernels in this file:
//   assemble_fast_kernel   triangles (the timed path): two threads per node, one 16-byte "fast record"
//                          per (visit, scalar row) with every address resolved at plan time, diagonal and
//                          fan-edge columns carried in registers, L2 prefetch of the next wave's records;
//                          damaged cells (d > 0) copy the row slices of per-cell element tangents
//                          (cell_setup_damage_kernel);
//   assemble_kernel        the generic-record form: Q2 and assembly_path = 2 (per-quadrature-point
//                          integration per visit) and plans without fast records;
//   dirichlet_kernel, fro / trace kernels, the fused-norm correction kernels.
#include <cuda.h>  // CUtensorMap (type and enums only: cuTensorMapEncodeTiled is fetched through the runtime)

#include <algorithm>

#include "constitutive.cuh"
#include "element.cuh"
#include "plan.cuh"
#include "reduce.cuh"
#include "tma.cuh"

namespace femb {

// ---- tensor maps of the value array (host) -----------------------------------------------------------
// cuTensorMapEncodeTiled comes from the driver through the runtime's entry-point query: libfemb200.so does not link
// libcuda.  The value array is described as rows of 128 bytes (16 doubles); a box is `rows` such lines, SWIZZLE_128B.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled()
{
   static EncodeTiledFn fn = nullptr;
   static bool tried = false;
   if (!tried)
   {
      tried = true;
      void *p = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) == cudaSuccess &&
          q == cudaDriverEntryPointSuccess)
         fn = reinterpret_cast<EncodeTiledFn>(p);
      else
         cudaGetLastError();
   }
   return fn;
}

// Swizzle of the tile image (16-byte chunk index ^= 128-byte line index & mask): the TMA pattern that gives the fewest
// bank conflicts for the staging stores of the element family (tools/swizzle_sim.py): P2 rows (19 / 9 blocks) want
// SWIZZLE_128B (mask 7: 1.56 x the ideal wavefronts; 64B: 1.83, 32B: 2.97), P1 rows (7 blocks = 14 units per node, which
// SWIZZLE_128B folds onto two bank groups: 3.3 x) want SWIZZLE_32B (mask 1: 1.0 x).
template <int ET>
__host__ __device__ constexpr uint32_t image_swizzle_mask()
{
   return ET == FEMB200_P1 ? 1u : 7u;
}

// fills the plan's tensor maps for this value array (boxes of 8 lines and of 1 line of 128 bytes; 64-line boxes were
// measured 3 % slower on P2); false when tensor bulk
// stores cannot be used (the caller falls back to the store loop): no driver entry point, or a value array that does
// not start on a 128-byte line.  SWIZZLE_128B: the array as rows of 16 doubles; SWIZZLE_32B: as rows of 4 doubles (a
// 128-byte line = 4 rows).
static bool values_tensor_maps(femb200_plan *pm, double *d_values)
{
   if (pm->tmap_values == d_values) return true;
   EncodeTiledFn enc = encode_tiled();
   if (!enc || (reinterpret_cast<uintptr_t>(d_values) & 127) != 0) return false;
   const bool narrow = pm->etype == FEMB200_P1;                      // 32-byte rows
   const cuuint32_t rowd = narrow ? 4u : 16u, rpl = narrow ? 4u : 1u;  // doubles per row, rows per 128-byte line
   const cuuint64_t lines = (cuuint64_t)((4 * pm->nnzb + 15) / 16);  // 128-byte lines of the value array
   if (lines == 0 || lines * rpl >= ((cuuint64_t)1 << 31)) return false;  // row coordinates are 32-bit
   const cuuint64_t gdim[2] = {rowd, lines * rpl};
   const cuuint64_t gstride[1] = {rowd * 8};
   const cuuint32_t estride[2] = {1, 1};
   std::lock_guard<std::mutex> lock(pm->range_mtx);
   for (int k = 0; k < 2; ++k)
   {
      const cuuint32_t box[2] = {rowd, (k == 0 ? 8u : 1u) * rpl};
      CUtensorMap *tm = reinterpret_cast<CUtensorMap *>(pm->tmap[k]);
      if (enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, d_values, gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
              narrow ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      {
         pm->tmap_values = nullptr;
         return false;
      }
   }
   pm->tmap_values = d_values;
   return true;
}

__device__ __forceinline__ void stage_put(double2 *sv, int unit, double a, double b, bool first)
{
   double2 *p = sv + swz(unit);
   if (first)
      *p = make_double2(a, b);
   else
   {
      double2 v = *p;
      v.x += a;
      v.y += b;
      *p = v;
   }
}

// one 2x2 block into (row0 unit base r0, row1 unit base r1), slot s
__device__ __forceinline__ void stage_block(double2 *sv, int r0, int r1, int s, const double *k, bool first)
{
   stage_put(sv, r0 + s, k[0], k[1], first);
   stage_put(sv, r1 + s, k[2], k[3], first);
}

// W^{cd} for Hooke: |T| (lam g_c (x) g_d + mu g_d (x) g_c + mu (g_c . g_d) I)
__device__ __forceinline__ void w_block(const double *gc, const double *gd, double tl, double tm, double *w)
{
   const double xx = gc[0] * gd[0], yy = gc[1] * gd[1], xy = gc[0] * gd[1], yx = gc[1] * gd[0];
   w[0] = (tl + 2. * tm) * xx + tm * yy;
   w[1] = tl * xy + tm * yx;
   w[2] = tl * yx + tm * xy;
   w[3] = (tl + 2. * tm) * yy + tm * xx;
}

struct AsmArgs
{
   int64_t nnodes;
   const int32_t *nptr;
   const VisitRec *vrec;
   const uint4 *frec;
   const uint8_t *tcnt;
   const TileHdr *thdr;
   int flevels;  // levels (visits per node) of the fixed-stride fast-record layout
   int prefetch_tiles;  // record prefetch distance in tiles (0: off)
   const uint8_t *perm;
   const uint16_t *voff;
   const int64_t *brp;
   const int32_t *xdofmap, *dofmap;
   const double *x;
   int xs;
   const double *E;
   LameCoef lc;
   const double *dnod, *u;
   const double *cellrec;
   const double *celld;  // records of the damaged cells (see cell_setup_damage_kernel)
   const int32_t *tdam;  // [ntiles][dmg_stage_cap]: cell whose damage record goes to slot s of the tile's stage, -1: none
                         // (written by cell_setup_damage_kernel on every assembly through the plan's cell -> slot map)
   int variant;
   double *values;
   int stage_units;  // capacity of the staging image in 16-byte units (multiple of 8)
   int use_tma;      // fast kernel: the finished tile leaves with tensor bulk stores
};

// ---- fast path: straight-sided P1 / P2 triangle, linear elasticity --------------
// The three dependent load levels of a visit (visit record -> cell vertices ->
// coordinates) are split into separate functions so that the kernel can issue each
// level for a batch of visits before consuming any of them.
struct FastGeo
{
   double g1x, g1y, g2x, g2y;  // sqrt(|T| E) grad lambda_1, sqrt(|T| E) grad lambda_2 (original vertex order)
};

// per-cell pre-pass (coalesced over cells): everything a visit needs from its cell in
// one 48-byte record, so that a visit costs three 16-byte loads of one line instead
// of ten scattered 4/8-byte loads (the L1 tag stage, one line per cycle, was the
// throughput limit of the gather: profiles/r1_assemble_v3.md)
__global__ void cell_setup_kernel(int64_t ncells, const int32_t *__restrict__ xdofmap, const double *__restrict__ x,
                                  int xs, const double *__restrict__ E, LameCoef lc, double *__restrict__ rec)
{
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (e >= ncells) return;
   const int64_t v0 = xdofmap[3 * e], v1 = xdofmap[3 * e + 1], v2 = xdofmap[3 * e + 2];
   const double x0 = x[v0 * xs], y0 = x[v0 * xs + 1];
   const double x1 = x[v1 * xs], y1 = x[v1 * xs + 1];
   const double x2 = x[v2 * xs], y2 = x[v2 * xs + 1];
   const double det = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0);
   const double id = 1. / det;
   // W^{cd} is bilinear in the gradients and linear in |T| E: fold sqrt(|T| E) into both gradients,
   // so that a cell is one 32-byte record (two 16-byte loads per visit)
   const double sc = sqrt(0.5 * fabs(det) * E[e]) * id;
   double2 *r = reinterpret_cast<double2 *>(rec + 4 * e);
   r[0] = make_double2((y2 - y0) * sc, -(x2 - x0) * sc);
   r[1] = make_double2(-(y1 - y0) * sc, (x1 - x0) * sc);
}

__device__ __forceinline__ int stored_position(int b, int a, int nd);

// ---- damaged cells (d > 0 at some quadrature point): per-cell pre-pass ------------------
// The tangent D_q (M.cc:736-872 closed form, or the dual-number Hessian M.cc:752-765) depends on the cell
// only, but the gather assembly visits every cell once per node and scalar row.  The pre-pass
// (cell_setup_damage_kernel) classifies the cells: undamaged ones keep the 32-byte fast-path record, damaged
// ones get a NaN marker there and a DAMAGE RECORD at celld[cell] (indexed by the cell id: no compaction):
//     [0..3]            grad lambda_1, grad lambda_2 (plain)
//     [4 + 6 q .. + 5]  upper triangle (00, 01, 02, 11, 12, 22) of w_q |det J| D_q, for the nq points of the rule
// (P1: 10 doubles in a 96-byte slot, P2: 22 doubles = 176 B in a 192-byte slot, against the 1152 B of a full element
// tangent; D_q is symmetric to rounding, its upper triangle is kept).  The constitutive evaluation -- the expensive, branchy part -- happens
// once per cell; a visit rebuilds its 2 x 2nd row slice from the record with ~90 FMAs: on a straight-sided
// triangle the P2 basis gradients at the points of the 3-point rule are fixed combinations of the grad lambda_c
// (L_k = 2/3 at point k, 1/6 elsewhere), so with c_q = row h of B_a(q) D_q (three numbers per point),
// C = sum_q c_q and S_v = sum_q 4 L_v(q) c_q = 2/3 C + 2 c_v:
//     vertex column v        (S_v - C)   contracted with grad lambda_v
//     edge column (p, r)      S_p contracted with grad lambda_r  +  S_r contracted with grad lambda_p
// (K[(a,h), (b,.)] = sum_q c_q B_b(q)^t, M.cc:699-704, 885-887).
template <int ET>
__device__ __forceinline__ void tri_ref_grads(int q, double (*dN)[2], double *phi, double &w2)
{  // reference gradients, vertex basis and 2 * weight at point q of the rule of element.cuh
   double xi, eta, w;
   quad_point<ET>(q, xi, eta, w);
   ref_grads<ET>(xi, eta, dN);
   phi[0] = 1. - xi - eta, phi[1] = xi, phi[2] = eta;
   w2 = 2. * w;
}

// global stride of a damage record in doubles (whole 32-byte sectors) and the bytes of it that carry data (what a
// tile stages in shared memory: an odd number of 16-byte units, so records at consecutive slots start in different
// bank groups)
template <int ET>
__host__ __device__ constexpr int dmg_rec_doubles()
{
   return ET == FEMB200_P1 ? 12 : 24;
}
template <int ET>
__host__ __device__ constexpr int dmg_rec_bytes()
{
   return ET == FEMB200_P1 ? 80 : 176;
}
constexpr int kDmgStageBytes = 144 * 176;  // record stage of a tile: 144 P2 records / 316 P1 records
template <int ET>
__host__ __device__ constexpr int dmg_stage_cap()
{
   return kDmgStageBytes / dmg_rec_bytes<ET>();
}

// One thread per cell.  The damage records leave through a per-warp shared-memory stage as whole 32-byte
// sectors (a thread storing its own 256-byte record would touch 8 lines per store instruction).
template <int ET>
__global__ void __launch_bounds__(128)
cell_setup_damage_kernel(int64_t ncells, const int32_t *__restrict__ xdofmap, const int32_t *__restrict__ dofmap,
                         const double *__restrict__ x, int xs, const double *__restrict__ E, LameCoef lc,
                         const double *__restrict__ dnod, const double *__restrict__ u, int variant,
                         double *__restrict__ rec, double *__restrict__ celld, const uint4 *__restrict__ cref,
                         int32_t *__restrict__ tdam, int cap, int *__restrict__ dmg_counter, int spec)
{
   constexpr int nd = Elem<ET>::nd, nq = Elem<ET>::nq, RS = dmg_rec_doubles<ET>(), STRIDE = RS + 2;
   __shared__ __align__(16) double stage[4][32 * STRIDE];
   const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
   const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   const bool active = e < ncells;
   const int64_t ec = active ? e : ncells - 1;
   const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + 32 * warp;
   const int64_t v0 = xdofmap[3 * ec], v1 = xdofmap[3 * ec + 1], v2 = xdofmap[3 * ec + 2];
   // the dof map is loaded with the vertex map, not behind the damage test: the chain of dependent global loads of a
   // damaged cell is (maps) -> (x, d, u) instead of (vertex map) -> (x, d) -> (dof map) -> (u); with `spec` (most cells
   // were damaged last time) the gather of u is issued before the test as well.  ncu of the round-2 pre-pass at 100 %
   // damaged cells: 4.3 long-scoreboard stall cycles per issued instruction at 16 warps per SM.
   int32_t dm[nd];
#pragma unroll
   for (int b = 0; b < nd; ++b) dm[b] = u ? dofmap[ec * nd + b] : 0;
   const double dv[3] = {dnod[v0], dnod[v1], dnod[v2]};
   const double xv[3][2] = {{x[v0 * xs], x[v0 * xs + 1]}, {x[v1 * xs], x[v1 * xs + 1]}, {x[v2 * xs], x[v2 * xs + 1]}};
   double ue[nd][2];
   if (spec && u)
   {
#pragma unroll
      for (int b = 0; b < nd; ++b)
      {
         const int64_t gd = 2 * (int64_t)dm[b];
         ue[b][0] = u[gd], ue[b][1] = u[gd + 1];
      }
   }
   const double det = (xv[1][0] - xv[0][0]) * (xv[2][1] - xv[0][1]) - (xv[2][0] - xv[0][0]) * (xv[1][1] - xv[0][1]);
   const double id = 1. / det;
   // d at the points of the rule: vertex basis values (2/3 at the point's own vertex, 1/6 elsewhere; P1: the centroid)
   double dq[nq];
   bool damaged = false;
#pragma unroll
   for (int q = 0; q < nq; ++q)
   {
      double dN[nd][2], phi[3], w2;
      tri_ref_grads<ET>(q, dN, phi, w2);
      dq[q] = phi[0] * dv[0] + phi[1] * dv[1] + phi[2] * dv[2];
      damaged = damaged || dq[q] > 0.;
   }
   damaged = damaged && active;
   const double g1x = (xv[2][1] - xv[0][1]) * id, g1y = -(xv[2][0] - xv[0][0]) * id;
   const double g2x = -(xv[1][1] - xv[0][1]) * id, g2y = (xv[1][0] - xv[0][0]) * id;
   const double Ee = E[ec];
   if (active)
   {
      double2 *r = reinterpret_cast<double2 *>(rec + 4 * e);
      if (!damaged)
      {  // the fast-path record of cell_setup_kernel
         const double sc = sqrt(0.5 * fabs(det) * Ee);
         r[0] = make_double2(g1x * sc, g1y * sc);
         r[1] = make_double2(g2x * sc, g2y * sc);
      }
      else
      {  // NaN marker: the damage record of this cell is celld[e]
         r[0] = make_double2(__longlong_as_double(0x7ff8000000000000ll), 0.);
         r[1] = make_double2(0., 0.);
      }
   }
   if (active && cref)
   {  // tell every tile that stages this cell (plan: tile << 10 | slot; slot 0x3ff: visited, not staged) whether the slot
      // holds a damaged cell this time
      const uint4 ra = cref[2 * e], rb = cref[2 * e + 1];
      const uint32_t ref[6] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y};
#pragma unroll
      for (int k = 0; k < 6; ++k)
         if (ref[k] != 0xffffffffu && (ref[k] & 0x3ffu) != 0x3ffu)
            tdam[(int64_t)(ref[k] >> 10) * cap + (ref[k] & 0x3ffu)] = damaged ? (int32_t)e : -1;
   }
   double *R = stage[warp] + lane * STRIDE;
   if (damaged)
   {
      R[0] = g1x, R[1] = g1y, R[2] = g2x, R[3] = g2y;
      const double lam = Ee * lc.c2, mu = Ee * lc.c3;
      if (!(spec && u))
      {
#pragma unroll
         for (int b = 0; b < nd; ++b)
         {
            if (u)
            {
               const int64_t gd = 2 * (int64_t)dm[b];
               ue[b][0] = u[gd], ue[b][1] = u[gd + 1];
            }
            else
               ue[b][0] = ue[b][1] = 0.;
         }
      }
      // straight-sided triangle: J is constant, so grad u at a point is sum_k t_k (x) grad lambda_k with
      // t_k = (4 L_k - 1) u_k + 4 sum over the edges at vertex k of L_(other end) u_edge  (P1: t_k = u_k), and with
      // grad lambda_0 = -(grad lambda_1 + grad lambda_2):  grad u = (t_1 - t_0) (x) g1 + (t_2 - t_0) (x) g2
      // (the same numbers as u_b G_b of M.cc:742 with G = dN J^-1, M.cc:696, without the per-point inverse)
      const double wq = (ET == FEMB200_P1 ? 0.5 : 1. / 6.) * fabs(det);
#pragma unroll 1
      for (int q = 0; q < nq; ++q)
      {
         double D[9];
         if (dq[q] > 0.)
         {
            double t[3][2];
            if (ET == FEMB200_P1)
            {
#pragma unroll
               for (int k = 0; k < 3; ++k) t[k][0] = ue[k][0], t[k][1] = ue[k][1];
            }
            else
            {
               const double L0 = q == 0 ? 2. / 3. : 1. / 6., L1 = q == 1 ? 2. / 3. : 1. / 6., L2 = q == 2 ? 2. / 3. : 1. / 6.;
#pragma unroll
               for (int c = 0; c < 2; ++c)
               {  // edge 3 + i is opposite vertex i
                  t[0][c] = (4. * L0 - 1.) * ue[0][c] + 4. * (L2 * ue[nd > 3 ? 4 : 0][c] + L1 * ue[nd > 3 ? 5 : 0][c]);
                  t[1][c] = (4. * L1 - 1.) * ue[1][c] + 4. * (L2 * ue[nd > 3 ? 3 : 0][c] + L0 * ue[nd > 3 ? 5 : 0][c]);
                  t[2][c] = (4. * L2 - 1.) * ue[2][c] + 4. * (L1 * ue[nd > 3 ? 3 : 0][c] + L0 * ue[nd > 3 ? 4 : 0][c]);
               }
            }
            const double a0 = t[1][0] - t[0][0], a1 = t[1][1] - t[0][1], b0 = t[2][0] - t[0][0], b1 = t[2][1] - t[0][1];
            const double g00 = a0 * g1x + b0 * g2x, g01 = a0 * g1y + b0 * g2y;  // grad u (M.cc:742)
            const double g10 = a1 * g1x + b1 * g2x, g11 = a1 * g1y + b1 * g2y;
            const double sh = 0.5 * (g01 + g10);
            const double eps[4] = {g00, sh, sh, g11};
            tangent(variant, lam, mu, dq[q], eps, D);
         }
         else
            hooke_scaled(lam, mu, 1., D);
         double *Rq = R + 4 + 6 * q;
         Rq[0] = D[0] * wq, Rq[1] = D[1] * wq, Rq[2] = D[2] * wq, Rq[3] = D[4] * wq, Rq[4] = D[5] * wq, Rq[5] = D[8] * wq;
      }
#pragma unroll
      for (int k = 4 + 6 * nq; k < RS; ++k) R[k] = 0.;
   }
   const unsigned mask = __ballot_sync(0xffffffffu, damaged);
   if (lane == 0 && mask && dmg_counter) atomicAdd(dmg_counter, __popc(mask));  // damaged cells of this assembly
   __syncwarp();
   constexpr int UPC = RS / 2;  // 16-byte units per record
   for (int t = lane; t < 32 * UPC; t += 32)
   {
      const int c = t / UPC, k = t - c * UPC;
      if ((mask >> c) & 1u)
         reinterpret_cast<double2 *>(celld + (e0 + c) * RS)[k] = reinterpret_cast<const double2 *>(stage[warp] + c * STRIDE)[k];
   }
}

// symmetric D of one point from a damage record
struct SymD
{
   double d00, d01, d02, d11, d12, d22;
};
__device__ __forceinline__ SymD ld_symd(const double *p)
{  // three 16-byte loads; p may point into the tile's record stage (shared) or into celld (global)
   const double2 a = *reinterpret_cast<const double2 *>(p), b = *reinterpret_cast<const double2 *>(p + 2),
                 c = *reinterpret_cast<const double2 *>(p + 4);
   SymD D;
   D.d00 = a.x, D.d01 = a.y, D.d02 = b.x, D.d11 = b.y, D.d12 = c.x, D.d22 = c.y;
   return D;
}
__device__ __forceinline__ void ld_grads(const double *p, double &g1x, double &g1y, double &g2x, double &g2y)
{
   const double2 a = *reinterpret_cast<const double2 *>(p), b = *reinterpret_cast<const double2 *>(p + 2);
   g1x = a.x, g1y = a.y, g2x = b.x, g2y = b.y;
}
// row h of B_a D with B rows (a,0) = [Gx, 0, Gy], (a,1) = [0, Gy, Gx]  (M.cc:699-704)
__device__ __forceinline__ void bd_row(const SymD &D, double gx, double gy, int h, double *c)
{
   const double p0 = h ? gy : gx, p2 = h ? gx : gy;  // multiply D row h and D row 2
   c[0] = p0 * (h ? D.d01 : D.d00) + p2 * D.d02;
   c[1] = p0 * (h ? D.d11 : D.d01) + p2 * D.d12;
   c[2] = p0 * (h ? D.d12 : D.d02) + p2 * D.d22;
}
// (K[(a,h),(b,0)], K[(a,h),(b,1)]) += c contracted with B_b, gradient (gx, gy)
__device__ __forceinline__ void cb_add(const double *c, double gx, double gy, double &k0, double &k1)
{
   k0 += c[0] * gx + c[2] * gy;
   k1 += c[1] * gy + c[2] * gx;
}

// Row (a, h) of the element tangent of a damaged cell from its damage record, natural local numbering:
// k[b] = (K[(a,h), (b,0)], K[(a,h), (b,1)]).  The plain per-point form (fallback kernels).
template <int ET>
__device__ __forceinline__ void damaged_row_slice(const double *__restrict__ R, int a, int h, double (*k)[2])
{
   constexpr int nd = Elem<ET>::nd, nq = Elem<ET>::nq;
   double g[3][2];
   ld_grads(R, g[1][0], g[1][1], g[2][0], g[2][1]);
   g[0][0] = -g[1][0] - g[2][0], g[0][1] = -g[1][1] - g[2][1];
#pragma unroll
   for (int b = 0; b < nd; ++b) k[b][0] = k[b][1] = 0.;
#pragma unroll
   for (int q = 0; q < nq; ++q)
   {
      const SymD D = ld_symd(R + 4 + 6 * q);
      double G[nd][2];
      if (ET == FEMB200_P1)
      {
#pragma unroll
         for (int v = 0; v < 3; ++v) G[v][0] = g[v][0], G[v][1] = g[v][1];
      }
      else
      {  // P2 at point q of the 3-point rule: L_q = 2/3, the other two 1/6 (element.cuh)
#pragma unroll
         for (int v = 0; v < 3; ++v)
         {
            const double cv = (v == q) ? 5. / 3. : -1. / 3.;  // 4 L_v - 1
            G[v][0] = cv * g[v][0], G[v][1] = cv * g[v][1];
            const int p = (v + 1) % 3, r = (v + 2) % 3;         // the edge opposite v joins p and r
            const double Lp = (p == q) ? 2. / 3. : 1. / 6., Lr = (r == q) ? 2. / 3. : 1. / 6.;
            G[3 + v][0] = 4. * (Lp * g[r][0] + Lr * g[p][0]);
            G[3 + v][1] = 4. * (Lp * g[r][1] + Lr * g[p][1]);
         }
      }
      double gax = 0., gay = 0.;
#pragma unroll
      for (int b = 0; b < nd; ++b)
         if (b == a) gax = G[b][0], gay = G[b][1];
      double c[3];
      bd_row(D, gax, gay, h, c);
#pragma unroll
      for (int b = 0; b < nd; ++b) cb_add(c, G[b][0], G[b][1], k[b][0], k[b][1]);
   }
}

// row slice of a damaged cell staged by the visit-record kernel: scalar row h of local row a
template <int ET>
__device__ __forceinline__ void damaged_compute_stage(const AsmArgs &A, const Visit &r, double2 *sv, int rbase, int h)
{
   constexpr int nd = Elem<ET>::nd;
   const int a = r.a;
   double k[nd][2];
   damaged_row_slice<ET>(A.celld + (int64_t)r.e * dmg_rec_doubles<ET>(), a, h, k);
#pragma unroll
   for (int b = 0; b < nd; ++b)
   {
      const int t = stored_position(b, a, nd);
      stage_put(sv, rbase + r.slot(t), k[b][0], k[b][1], r.is_first(t));
   }
}

__device__ __forceinline__ FastGeo fast_geo(const AsmArgs &A, const Visit &r)
{
   FastGeo g;
   ld_d4(A.cellrec + 4 * (int64_t)r.e, g.g1x, g.g1y, g.g2x, g.g2y);
   return g;
}

// stored position (plan.cuh) of natural local dof b in the visit record of a row with local index a
__device__ __forceinline__ int stored_position(int b, int a, int nd)
{
   if (nd > 6) return b;
   const int m = (a >= 3) ? a - 3 : a;
   const int bb = (b >= 3) ? b - 3 : b;
   int tt = bb - m;
   tt = (tt < 0) ? tt + 3 : tt;
   return (b >= 3) ? tt + 3 : tt;
}

// row 0 of W^{cd} = |T| (lam g_c (x) g_d + mu g_d (x) g_c + mu (g_c . g_d) I)
__device__ __forceinline__ void w_row(const double *gc, const double *gd, double tl, double tm, double *w)
{
   w[0] = (tl + 2. * tm) * (gc[0] * gd[0]) + tm * (gc[1] * gd[1]);
   w[1] = tl * (gc[0] * gd[1]) + tm * (gc[1] * gd[0]);
}

// Computes ONE scalar row (h = 0: x-row, h = 1: y-row) of the row slice of the element
// matrix owned by the visit and stages it: two threads share a node, which doubles
// the resident warps for the same staging footprint.  Row 1 is row 0 with the x and y
// components of every gradient exchanged and the two outputs swapped.
template <int ET>
__device__ __forceinline__ void fast_compute_stage(const AsmArgs &A, const Visit &r, const FastGeo &g, double2 *sv,
                                                   int rbase, int h)
{
   const int a = r.a;
   const int m = (a >= 3) ? a - 3 : a;  // rotation: own vertex / own edge becomes number 0
   // gradients of the rotated barycentric coordinates 1' = m + 1, 2' = m + 2 (mod 3)
   const double h0x = -g.g1x - g.g2x, h0y = -g.g1y - g.g2y;
   const double a1x = m == 0 ? g.g1x : (m == 1 ? g.g2x : h0x), a1y = m == 0 ? g.g1y : (m == 1 ? g.g2y : h0y);
   const double a2x = m == 0 ? g.g2x : (m == 1 ? h0x : g.g1x), a2y = m == 0 ? g.g2y : (m == 1 ? h0y : g.g1y);
   const double g1[2] = {h ? a1y : a1x, h ? a1x : a1y};
   const double g2[2] = {h ? a2y : a2x, h ? a2x : a2y};
   const double tl = A.lc.c2, tm = A.lc.c3;
   double k[2];
   auto put = [&](int t, const double *kk) {
      stage_put(sv, rbase + r.slot(t), h ? kk[1] : kk[0], h ? kk[0] : kk[1], r.is_first(t));  // rotated order
   };
   if (a < 3)
   {  // row = (rotated) vertex 0
      const double g0[2] = {-g1[0] - g2[0], -g1[1] - g2[1]};
      double w00[2], w01[2], w02[2];
      w_row(g0, g0, tl, tm, w00);
      w_row(g0, g1, tl, tm, w01);
      w_row(g0, g2, tl, tm, w02);
      if (ET == FEMB200_P1)
      {  // P1: K_ab = W^{ab}  (M.cc:885-887)
         put(0, w00);
         put(1, w01);
         put(2, w02);
      }
      else
      {
         const double c3 = -1. / 3., c43 = 4. / 3.;
         put(0, w00);
         k[0] = c3 * w01[0], k[1] = c3 * w01[1];
         put(1, k);
         k[0] = c3 * w02[0], k[1] = c3 * w02[1];
         put(2, k);
         // rotated edges: 0' = (1,2) opposite (structural zero), 1' = (2,0), 2' = (0,1)
         k[0] = k[1] = 0.;
         put(3, k);
         k[0] = c43 * w02[0], k[1] = c43 * w02[1];
         put(4, k);
         k[0] = c43 * w01[0], k[1] = c43 * w01[1];
         put(5, k);
      }
   }
   else
   {  // row = (rotated) edge 0 = (1,2); uses sum_d W^{cd} = 0 to stay within W11, W12, W21, W22
      double w11[2], w12[2], w21[2], w22[2];
      w_row(g1, g1, tl, tm, w11);
      w_row(g1, g2, tl, tm, w12);
      w_row(g2, g1, tl, tm, w21);  // = row of (W^{12})^t
      w_row(g2, g2, tl, tm, w22);
      const double c43 = 4. / 3.;
      // vertices: opposite 0' -> 0; 1' (= p) -> 4/3 W^{21}; 2' (= q) -> 4/3 W^{12}
      k[0] = k[1] = 0.;
      put(0, k);
      k[0] = c43 * w21[0], k[1] = c43 * w21[1];
      put(1, k);
      k[0] = c43 * w12[0], k[1] = c43 * w12[1];
      put(2, k);
      const double sy[2] = {w12[0] + w21[0], w12[1] + w21[1]};  // S = W12 + W21
      k[0] = c43 * (2. * w11[0] + sy[0] + 2. * w22[0]), k[1] = c43 * (2. * w11[1] + sy[1] + 2. * w22[1]);
      put(3, k);
      k[0] = -c43 * (2. * w11[0] + sy[0]), k[1] = -c43 * (2. * w11[1] + sy[1]);
      put(4, k);
      k[0] = -c43 * (sy[0] + 2. * w22[0]), k[1] = -c43 * (sy[1] + 2. * w22[1]);
      put(5, k);
   }
}

// The row-slice computation driven by a fast-path record (plan.cuh): the staging address and the
// first-touch bit of every column come out of the record with one or two integer operations; the
// diagonal block is accumulated in registers (dg) and the two columns shared with the next visit of
// the fan are carried in registers (cv, ce) instead of going through the staging image.
struct FastCarry
{
   double dg[2], cv[2], ce[2];
};

// fields of a fast-path record (plan.cuh): ONE record per visit, shared by the two scalar-row threads of the node
__device__ __forceinline__ int rec_i1(const uint4 r) { return (int)((r.y >> 29) & 3u); }
__device__ __forceinline__ int rec_i2(const uint4 r) { return (int)((r.z >> 29) & 3u); }
__device__ __forceinline__ bool rec_edge(const uint4 r) { return (r.y >> 28) & 1u; }
__device__ __forceinline__ bool rec_cout(const uint4 r) { return (r.y >> 27) & 1u; }
__device__ __forceinline__ bool rec_first(const uint4 r, int b) { return (r.y >> (22 + b)) & 1u; }
// units between the two scalar rows of the node in the image (its block degree), times h
__device__ __forceinline__ uint32_t rec_hdeg(const uint4 r, int h) { return h ? ((r.z >> 22) & 0x7fu) : 0u; }
// byte offset in the tile image of column t (position t of the record) of scalar row h: position of row 0 + h deg,
// chunk-swizzled inside its 128-byte line (swz_tma)
template <uint32_t MASK>
__device__ __forceinline__ uint32_t rec_off(const uint4 r, int t, uint32_t hdeg)
{
   const uint32_t w = t < 2 ? r.y : (t < 4 ? r.z : r.w);
   const uint32_t p = (((t & 1) ? (w >> 11) : w) & 0x7ffu) + hdeg;
   return (p ^ ((p >> 3) & MASK)) << 4;
}

// Values of the row slice of one visit, positions t = 0..5 of the record's numbering (0', 1', 2', then
// the edges opposite to them), for scalar row h, in the EXCHANGED frame of row h: for h = 1 the two
// entries of every pair are swapped (row 1 of the closed form is row 0 with x and y exchanged in every
// gradient and every output pair); emit_row_slice() swaps them back when it stores.
template <int ET, bool EDGE>
__device__ __forceinline__ void fast_values(const AsmArgs &A, const uint4 raw, const FastGeo &g, int h, double (*v)[2])
{
   // gradients of the visit's vertices 1' and 2' (local numbers from the record; 0' is the row's own
   // vertex, or the vertex opposite to the row's own edge)
   const int i1 = rec_i1(raw), i2 = rec_i2(raw);
   const double h0x = -g.g1x - g.g2x, h0y = -g.g1y - g.g2y;
   const double a1x = i1 == 0 ? h0x : (i1 == 1 ? g.g1x : g.g2x), a1y = i1 == 0 ? h0y : (i1 == 1 ? g.g1y : g.g2y);
   const double a2x = i2 == 0 ? h0x : (i2 == 1 ? g.g1x : g.g2x), a2y = i2 == 0 ? h0y : (i2 == 1 ? g.g1y : g.g2y);
   const double g1[2] = {h ? a1y : a1x, h ? a1x : a1y};
   const double g2[2] = {h ? a2y : a2x, h ? a2x : a2y};
   const double tl = A.lc.c2, tm = A.lc.c3;
   if (!EDGE)
   {  // row = vertex 0'
      const double g0[2] = {-g1[0] - g2[0], -g1[1] - g2[1]};
      double w01[2], w02[2];
      w_row(g0, g0, tl, tm, v[0]);
      w_row(g0, g1, tl, tm, w01);
      w_row(g0, g2, tl, tm, w02);
      // P1: K_ab = W^{ab} (M.cc:885-887); P2: vertex / vertex -1/3 W, vertex / adjacent edge 4/3 W,
      // vertex / opposite edge 0
      const double c3 = ET == FEMB200_P1 ? 1. : -1. / 3., c43 = 4. / 3.;
      v[1][0] = c3 * w01[0], v[1][1] = c3 * w01[1];
      v[2][0] = c3 * w02[0], v[2][1] = c3 * w02[1];
      if (ET != FEMB200_P1)
      {
         v[3][0] = v[3][1] = 0.;
         v[4][0] = c43 * w02[0], v[4][1] = c43 * w02[1];
         v[5][0] = c43 * w01[0], v[5][1] = c43 * w01[1];
      }
   }
   else
   {  // row = edge 0' = (1', 2'); uses sum_d W^{cd} = 0 to stay within W11, W12, W21, W22
      double w11[2], w12[2], w21[2], w22[2];
      w_row(g1, g1, tl, tm, w11);
      w_row(g1, g2, tl, tm, w12);
      w_row(g2, g1, tl, tm, w21);  // = row of (W^{12})^t
      w_row(g2, g2, tl, tm, w22);
      const double c43 = 4. / 3.;
      const double sy[2] = {w12[0] + w21[0], w12[1] + w21[1]};  // S = W12 + W21
      v[0][0] = v[0][1] = 0.;  // opposite vertex
      v[1][0] = c43 * w21[0], v[1][1] = c43 * w21[1];
      v[2][0] = c43 * w12[0], v[2][1] = c43 * w12[1];
      v[3][0] = c43 * (2. * w11[0] + sy[0] + 2. * w22[0]), v[3][1] = c43 * (2. * w11[1] + sy[1] + 2. * w22[1]);
      v[4][0] = -c43 * (2. * w11[0] + sy[0]), v[4][1] = -c43 * (2. * w11[1] + sy[1]);
      v[5][0] = -c43 * (sy[0] + 2. * w22[0]), v[5][1] = -c43 * (sy[1] + 2. * w22[1]);
   }
}

// The same slice for a damaged cell, rebuilt from the cell's damage record in the record's own frame: positions
// 0', 1', 2' are the local vertices i0, i1, i2 (i0 = the row's vertex, or the vertex opposite to the row's edge),
// positions 3..5 the edges opposite to them; the point of the rule that sits next to vertex i_t is "point t".
template <int ET, bool EDGE>
__device__ __forceinline__ void damaged_values(const double *R, const uint4 raw, int h, double (*v)[2])
{
   const int i1 = rec_i1(raw), i2 = rec_i2(raw), i0 = 3 - i1 - i2;
   double g1x, g1y, g2x, g2y;
   ld_grads(R, g1x, g1y, g2x, g2y);
   const double h0x = -g1x - g2x, h0y = -g1y - g2y;
   // gradients of lambda at positions 1', 2', 0'
   const double p1x = i1 == 0 ? h0x : (i1 == 1 ? g1x : g2x), p1y = i1 == 0 ? h0y : (i1 == 1 ? g1y : g2y);
   const double p2x = i2 == 0 ? h0x : (i2 == 1 ? g1x : g2x), p2y = i2 == 0 ? h0y : (i2 == 1 ? g1y : g2y);
   const double p0x = -p1x - p2x, p0y = -p1y - p2y;
   auto out = [&](int t, double k0, double k1) { v[t][0] = h ? k1 : k0, v[t][1] = h ? k0 : k1; };  // exchanged frame
   if (ET == FEMB200_P1)
   {  // one point, constant gradients: K_ab = (row h of B_a D) B_b^t
      const SymD D = ld_symd(R + 4);
      double c[3];
      bd_row(D, p0x, p0y, h, c);
      double k0, k1;
      k0 = k1 = 0., cb_add(c, p0x, p0y, k0, k1), out(0, k0, k1);
      k0 = k1 = 0., cb_add(c, p1x, p1y, k0, k1), out(1, k0, k1);
      k0 = k1 = 0., cb_add(c, p2x, p2y, k0, k1), out(2, k0, k1);
      return;
   }
   // D at the points next to 0', 1', 2' (point index = local vertex number)
   const SymD D0 = ld_symd(R + 4 + 6 * i0), D1 = ld_symd(R + 4 + 6 * i1), D2 = ld_symd(R + 4 + 6 * i2);
   // c_t = row h of B_a(point t) D_t: gradient of the row's own basis function at the three points
   double c0[3], c1[3], c2[3];
   if (!EDGE)
   {  // vertex 0': (4 L_0 - 1) grad lambda_0 = 5/3, -1/3, -1/3
      bd_row(D0, (5. / 3.) * p0x, (5. / 3.) * p0y, h, c0);
      bd_row(D1, (-1. / 3.) * p0x, (-1. / 3.) * p0y, h, c1);
      bd_row(D2, (-1. / 3.) * p0x, (-1. / 3.) * p0y, h, c2);
   }
   else
   {  // edge (1', 2'): 4 (L_1 grad lambda_2 + L_2 grad lambda_1)
      bd_row(D0, (-2. / 3.) * p0x, (-2. / 3.) * p0y, h, c0);
      bd_row(D1, (8. / 3.) * p2x + (2. / 3.) * p1x, (8. / 3.) * p2y + (2. / 3.) * p1y, h, c1);
      bd_row(D2, (2. / 3.) * p2x + (8. / 3.) * p1x, (2. / 3.) * p2y + (8. / 3.) * p1y, h, c2);
   }
   double S0[3], S1[3], S2[3], P0[3], P1[3], P2[3];
#pragma unroll
   for (int j = 0; j < 3; ++j)
   {
      const double C = c0[j] + c1[j] + c2[j];
      S0[j] = (2. / 3.) * C + 2. * c0[j], S1[j] = (2. / 3.) * C + 2. * c1[j], S2[j] = (2. / 3.) * C + 2. * c2[j];
      P0[j] = S0[j] - C, P1[j] = S1[j] - C, P2[j] = S2[j] - C;
   }
   double k0, k1;
   k0 = k1 = 0., cb_add(P0, p0x, p0y, k0, k1), out(0, k0, k1);
   k0 = k1 = 0., cb_add(P1, p1x, p1y, k0, k1), out(1, k0, k1);
   k0 = k1 = 0., cb_add(P2, p2x, p2y, k0, k1), out(2, k0, k1);
   // edge opposite t joins the other two positions
   k0 = k1 = 0., cb_add(S1, p2x, p2y, k0, k1), cb_add(S2, p1x, p1y, k0, k1), out(3, k0, k1);
   k0 = k1 = 0., cb_add(S0, p2x, p2y, k0, k1), cb_add(S2, p0x, p0y, k0, k1), out(4, k0, k1);
   k0 = k1 = 0., cb_add(S0, p1x, p1y, k0, k1), cb_add(S1, p0x, p0y, k0, k1), out(5, k0, k1);
}

// Accumulates / carries / stages the slice: the diagonal block goes to registers (C.dg); the carry
// registers are added to side 0; side 1 is carried when the record says so (plan.cu, k_fast_records).
template <int ET, bool EDGE>
__device__ __forceinline__ void emit_row_slice(const uint4 raw, unsigned char *sv, int h, FastCarry &C,
                                               const double (*v)[2])
{
   const bool cout = rec_cout(raw);
   const uint32_t hdeg = rec_hdeg(raw, h);
   // t = position (address entry), b = index of the put (first-touch bit)
   auto put = [&](int t, int b, double k0, double k1) {
      const uint32_t off = rec_off<image_swizzle_mask<ET>()>(raw, t, hdeg);
      const bool first = rec_first(raw, b);
      double2 *p = reinterpret_cast<double2 *>(sv + off);
      const double va = h ? k1 : k0, vb = h ? k0 : k1;
      if (first)
         *p = make_double2(va, vb);
      else
      {
         double2 x = *p;
         x.x += va, x.y += vb;
         *p = x;
      }
   };
   if (!EDGE)
   {  // vertex row: side 0 = positions (1, 5), side 1 = positions (2, 4)
      C.dg[0] += v[0][0], C.dg[1] += v[0][1];
      put(1, 0, v[1][0] + C.cv[0], v[1][1] + C.cv[1]);
      if (ET != FEMB200_P1)
      {
         put(5, 4, v[5][0] + C.ce[0], v[5][1] + C.ce[1]);
         put(3, 2, v[3][0], v[3][1]);
      }
      if (cout)
      {
         C.cv[0] = v[2][0], C.cv[1] = v[2][1];
         if (ET != FEMB200_P1) C.ce[0] = v[4][0], C.ce[1] = v[4][1];
      }
      else
      {
         put(2, 1, v[2][0], v[2][1]);
         if (ET != FEMB200_P1) put(4, 3, v[4][0], v[4][1]);
         C.cv[0] = C.cv[1] = C.ce[0] = C.ce[1] = 0.;
      }
   }
   else
   {  // edge row: the two end columns (positions 1, 2) go from the first cell to the second
      C.dg[0] += v[3][0], C.dg[1] += v[3][1];
      put(0, 0, v[0][0], v[0][1]);
      put(4, 3, v[4][0], v[4][1]);
      put(5, 4, v[5][0], v[5][1]);
      const double v1[2] = {v[1][0] + C.cv[0], v[1][1] + C.cv[1]};
      const double v2[2] = {v[2][0] + C.ce[0], v[2][1] + C.ce[1]};
      if (cout)
         C.cv[0] = v1[0], C.cv[1] = v1[1], C.ce[0] = v2[0], C.ce[1] = v2[1];
      else
      {
         put(1, 1, v1[0], v1[1]);
         put(2, 2, v2[0], v2[1]);
         C.cv[0] = C.cv[1] = C.ce[0] = C.ce[1] = 0.;
      }
   }
}

// Fast kernel (undamaged triangles): two threads per node (one per scalar row: lanes 0-15 of a warp
// own row 0 of 16 nodes, lanes 16-31 row 1 of the same nodes), nodes ranked by decreasing visit
// count.  The records live in a fixed-stride layout (tile, level, rank, row), so their addresses
// depend on the block and thread index only: the dependent chain of a tile is record -> cell record
// -> first put (the tile header is needed by the stream-out only), with the cell record one visit
// and the record two visits ahead.
template <int ET, bool DMG, bool NORMS, int MINB, bool STAGE = false>
__global__ void __launch_bounds__(kAsmR * 2, MINB)
assemble_fast_kernel(AsmArgs A, ReduceScratch red, double *__restrict__ norms_out, const __grid_constant__ CUtensorMap tm8,
                     const __grid_constant__ CUtensorMap tm1)
{
   constexpr int R = kAsmR, THREADS = kAsmR * 2;
   extern __shared__ __align__(1024) double2 sv[];
   const int tid = threadIdx.x;
   const int64_t tile = blockIdx.x, ntiles = gridDim.x;
   unsigned char *dstage = reinterpret_cast<unsigned char *>(sv) + 16 * (size_t)A.stage_units;
   uint64_t *dbar = reinterpret_cast<uint64_t *>(dstage + kDmgStageBytes);
   if (STAGE)
   {
      if (tid == 0)
      {
         mbar_init(dbar, THREADS);
         asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      }
      __syncthreads();  // the barrier is initialised (nothing is in flight yet: all warps arrive at once)
   }
   const TileHdr *hdr = A.thdr + tile;
   const int64_t b0 = hdr->b0;
   const int units = hdr->units;  // 16-byte units of this tile
   const int rank = ((tid >> 5) << 4) + (tid & 15);
   const int half = (tid >> 4) & 1;
   double nrm[2] = {0., 0.};  // NORMS: this thread's share of sum v^2 and of the trace
   // DMG: the damage records of the tile's cells (plan list tcell, slot number in the fast records) are staged behind
   // the image with one bulk copy per damaged cell (no LSU instruction, no register): a visit then reads its record
   // with 16-byte shared-memory loads (the two row threads of a node read the same addresses: broadcast) instead of
   // pulling 176 bytes through L1 as scattered 32-byte sectors.
   // Fill of the stage: the tile's row of tdam says which slots hold a damaged cell this time; one 16-byte LDGSTS per
   // (slot, unit of the record), completion on the mbarrier.  The records of the tile `prefetch_tiles` ahead are
   // pulled into L2 (thread = (slot, 128-byte line)), its tdam row was prefetched by the tile that far behind.
   constexpr int DCAP = dmg_stage_cap<ET>(), DUPR = dmg_rec_bytes<ET>() / 16, DRS = dmg_rec_doubles<ET>();
   constexpr int DNR = STAGE ? (DCAP + THREADS - 1) / THREADS : 1;                 // row entries per thread
   constexpr int DNF = STAGE ? (DCAP * DUPR + THREADS - 1) / THREADS : 1;          // fill units per thread
   constexpr int DLPR = (DRS * 8 + 127) / 128;                                   // 128-byte lines per record
   const bool dstg = STAGE && A.tdam != nullptr;
   const bool dpf = dstg && A.prefetch_tiles > 0 && (int64_t)tile + A.prefetch_tiles < ntiles;
   int32_t *drow = reinterpret_cast<int32_t *>(dstage + kDmgStageBytes + 16);    // [DCAP] this tile's row of tdam
   int32_t rcell[DNR], fcell[DNR];
   if (STAGE)
   {
#pragma unroll
      for (int k = 0; k < DNR; ++k)
      {
         const int i = tid + k * THREADS;
         rcell[k] = (dstg && i < DCAP) ? A.tdam[(int64_t)tile * DCAP + i] : -1;
         fcell[k] = (dpf && i < DCAP) ? A.tdam[((int64_t)tile + A.prefetch_tiles) * DCAP + i] : -1;
      }
   }
   bool staged = !STAGE;  // STAGE: whether this thread has waited for the record stage
   {
      const uint4 *rec = A.frec + ((int64_t)tile * A.flevels * R + rank);  // shared by the node's two row threads
      constexpr int LS = R;  // records per level
      unsigned char *img = reinterpret_cast<unsigned char *>(sv);
      const uint4 none = make_uint4(0u, 0u, 0u, 0u);
      uint4 raw = none, raw1, raw2;
      FastGeo geo, geo1;
      FastCarry C;
      C.dg[0] = C.dg[1] = C.cv[0] = C.cv[1] = C.ce[0] = C.ce[1] = 0.;
      // The records are read once, from DRAM, at the head of every tile's dependent chain: the records of the
      // tile `prefetch_tiles` ahead (1.5 - 2 waves of resident CTAs) are pulled into L2; that tile's visit
      // count for this rank comes from the plan's byte table, loaded together with the first record.
      const bool pf = A.prefetch_tiles > 0 && (int64_t)tile + A.prefetch_tiles < ntiles;
      const int cfut = pf ? (int)A.tcnt[((int64_t)tile + A.prefetch_tiles) * R + rank] : 0;
      // ... and half that distance ahead the records are in L2 already: the first record of that tile is read (one row
      // thread per node) and the cell record of its first visit, the second link of that tile's chain, prefetched
      const int ph = A.prefetch_tiles >> 1;  // measured: 0.683 -> 0.673 ms at n = 1448
      uint32_t rfut = 0u;
      if (ph > 0 && half == 0 && (int64_t)tile + ph < ntiles) rfut = reinterpret_cast<const uint32_t *>(rec + (int64_t)ph * A.flevels * LS)[0];
      raw1 = rec[0];
      raw2 = A.flevels > 1 ? rec[LS] : none;
      const int cnt = (int)(raw1.x >> 28);  // visits of this row (0: padding)
      if (cfut > 0 && (tid & 23) == 0)
      {  // one lane per 128-byte line of records (8 ranks; the first of them has the largest visit count)
         const uint4 *nx = rec + (int64_t)A.prefetch_tiles * A.flevels * LS;
#pragma unroll
         for (int j = 0; j < 8; ++j)
            if (j < cfut) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + j * LS));
      }
      if (0 < cnt) ld_d4(A.cellrec + 4 * (int64_t)(raw1.x & 0x0fffffffu), geo1.g1x, geo1.g1y, geo1.g2x, geo1.g2y);
      if (STAGE)
      {  // issue the stage fill behind the first loads of the visit pipeline: the row goes through shared memory (one
         // global load per thread instead of one per fill unit; measured 4 % faster than per-thread row loads)
#pragma unroll
         for (int k = 0; k < DNR; ++k)
            if (tid + k * THREADS < DCAP) drow[tid + k * THREADS] = rcell[k];
         __syncthreads();
#pragma unroll
         for (int k = 0; k < DNF; ++k)
         {
            const int i = tid + k * THREADS;
            if (i < DCAP * DUPR)
            {
               const int sl = i / DUPR;
               const int32_t cc = drow[sl];
               if (cc >= 0) cp_async16(dstage + 16 * i, A.celld + (int64_t)cc * DRS + 2 * (i - sl * DUPR));
            }
         }
         asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(dbar)) : "memory");
         if (dpf && (int64_t)tile + 2 * A.prefetch_tiles < ntiles && tid < (DCAP * 4 + 127) / 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(A.tdam + ((int64_t)tile + 2 * A.prefetch_tiles) * DCAP) + 128 * tid));
      }
      // One visit: the row slice of cell (R.x & 0x0fffffff) with its cell record G.
      auto visit = [&](const uint4 &R, const FastGeo &G) {
         // damaged cell: NaN marker; STAGE: its damage record is in the tile's stage (slot in the record), or, where the
         // tile has more cells than the stage holds (slot 0x3ff) and in the kernel without a stage, at celld[cell]
         const bool dam = DMG && G.g1x != G.g1x;
         const double *drec = nullptr;
         if (dam)
         {
            if (!staged) mbar_wait(dbar, 0), staged = true;
            const uint32_t slot = STAGE ? R.w >> 22 : 0x3ffu;
            drec = slot != 0x3ffu ? reinterpret_cast<const double *>(dstage + slot * dmg_rec_bytes<ET>())
                                  : A.celld + (int64_t)(R.x & 0x0fffffffu) * dmg_rec_doubles<ET>();
         }
         if (!rec_edge(R))
         {  // vertex row
            double v[Elem<ET>::nd][2];
            if (dam)
            {
               damaged_values<ET, false>(drec, R, half, v);
               emit_row_slice<ET, false>(R, img, half, C, v);
            }
            else
            {
               fast_values<ET, false>(A, R, G, half, v);
               emit_row_slice<ET, false>(R, img, half, C, v);
            }
         }
         else if (ET != FEMB200_P1)
         {  // edge row
            double v[Elem<ET>::nd][2];
            if (dam)
            {
               damaged_values<ET, true>(drec, R, half, v);
               emit_row_slice<ET, true>(R, img, half, C, v);
            }
            else
            {
               fast_values<ET, true>(A, R, G, half, v);
               emit_row_slice<ET, true>(R, img, half, C, v);
            }
         }
      };
      auto ld_geo = [&](const uint4 &R, FastGeo &G) { ld_d4(A.cellrec + 4 * (int64_t)(R.x & 0x0fffffffu), G.g1x, G.g1y, G.g2x, G.g2y); };
      // (Three named register sets used round robin with the loop unrolled by three would remove the 16 register moves
      // per visit of this rotation -- 14 % of the kernel's instructions are IMAD.MOV -- but spills at the 72 registers
      // of 7 CTAs per SM: 0.669 -> 1.165 ms at n = 1448; a carry flag as a 0 / 1 multiplier instead of the conditional
      // zeroing of the carry registers, another 16 moves per visit: 0.669 -> 0.703 ms; profiles/r2_experiments.md.)
      for (int c = 0; c < cnt; ++c)
      {
         raw = raw1, geo = geo1, raw1 = raw2;
         if (c + 1 < cnt) ld_geo(raw1, geo1);
         raw2 = (c + 2 < cnt) ? rec[(c + 2) * LS] : none;
         visit(raw, geo);
      }
      if (STAGE)
      {  // L2 prefetch of the damage records of the future tile
#pragma unroll
         for (int k = 0; k < DNR; ++k)
            if (fcell[k] >= 0)
            {
               const char *q = reinterpret_cast<const char *>(A.celld + (int64_t)fcell[k] * DRS);
#pragma unroll
               for (int l = 0; l < DLPR; ++l) asm volatile("prefetch.global.L2 [%0];" ::"l"(q + 128 * l));
            }
      }
      if ((rfut >> 28) != 0u) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.cellrec + 4 * (int64_t)(rfut & 0x0fffffffu)));
      if (cnt > 0)
      {  // the diagonal block, written once: position 0 of a vertex row, 3 of an edge row
         const uint32_t off = rec_off<image_swizzle_mask<ET>()>(raw, rec_edge(raw) ? 3 : 0, rec_hdeg(raw, half));
         *reinterpret_cast<double2 *>(img + off) = make_double2(half ? C.dg[1] : C.dg[0], half ? C.dg[0] : C.dg[1]);
         nrm[1] = C.dg[0];  // the diagonal entry of this scalar row (exchanged frame: first of the pair)
      }
   }
   __syncthreads();
   // Stream the finished tile out: one contiguous byte range of the CSR values.  Image position p holds the unit
   // (first unit of the tile - shift) + p of the value array, chunk-swizzled inside its 128-byte line (swz_tma).
   const int shift = (int)((2 * b0) & 7);
   const int end = shift + units;                                  // positions [shift, end) are this tile's
   double2 *dst = reinterpret_cast<double2 *>(A.values) + (2 * b0 - shift);  // position p <-> dst[p]
   if (!NORMS && A.use_tma)
   {
      // full lines [lf, ll) by the TMA unit (it reads shared memory itself and undoes the swizzle: no LDS, no STG,
      // no per-thread loop); the partial first / last line by 16 threads
      const int lf = shift ? 1 : 0, ll = end >> 3;
      constexpr int RPL = ET == FEMB200_P1 ? 4 : 1;  // tensor rows per 128-byte line (SWIZZLE_32B: 32-byte rows)
      if (tid == 0)
      {
         asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the image was written by ordinary stores
         const int gl0 = (int)((2 * b0 - shift) >> 3);                 // 128-byte line of the value array of image line 0
         int l = lf;
         for (; l + 8 <= ll; l += 8)
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(&tm8), "r"(0),
                         "r"((gl0 + l) * RPL), "r"(smem_u32(sv + 8 * l))
                         : "memory");
         for (; l < ll; ++l)
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(&tm1), "r"(0),
                         "r"((gl0 + l) * RPL), "r"(smem_u32(sv + 8 * l))
                         : "memory");
         asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      else if (tid >= 32 && tid < 48)
      {
         const int c = tid & 7, l = (tid < 40) ? 0 : ll;              // chunk, image line (first / last)
         const int p = 8 * l + (c ^ (l & (int)image_swizzle_mask<ET>()));
         const bool mine = (tid < 40) ? (shift != 0 && ll > 0) : ((end & 7) != 0);
         if (mine && p >= shift && p < end) st_stream_d2(reinterpret_cast<double *>(dst + p), sv[8 * l + c]);
      }
      if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the image must outlive the reads
   }
   else
   {
      // store loop.  The swizzle key of position q is (q >> 3) & 7, which the stride of THREADS = 16 lines leaves
      // alone: per thread the swizzle is one constant XOR.
      static_assert(THREADS % 64 == 0, "the stream-out stride must keep (q >> 3) & 7");
      const int kx = (tid >> 3) & (int)image_swizzle_mask<ET>();
      const int padded = (end + 7) & ~7;
      for (int q = tid; q < padded; q += THREADS)
      {
         const int p = q ^ kx;
         if (p >= shift && p < end)
         {
            const double2 val = sv[q];
            st_stream_d2(reinterpret_cast<double *>(dst + p), val);
            if (NORMS) nrm[0] += val.x * val.x + val.y * val.y;
         }
      }
   }
   // fused (|K|_F^2, trace K) of the unconstrained matrix: one partial pair per CTA, summed in a fixed
   // order by norms_sum_kernel
   if (NORMS)
   {
      __shared__ double sh[THREADS / 32];
      const double f2 = block_sum<THREADS>(nrm[0], sh), tr = block_sum<THREADS>(nrm[1], sh);
      if (tid == 0) red.partials[tile] = f2, red.partials[(size_t)ntiles + tile] = tr;
   }
}

// damaged cells of this assembly (counted by the pre-pass) -> host-mapped word, read without synchronisation by the
// NEXT damaged assembly on the plan to choose the kernel; the counter is cleared for the next pre-pass
__global__ void dmg_count_publish_kernel(int *__restrict__ counter, int *__restrict__ out)
{
   *out = *counter;
   *counter = 0;
}

__global__ void __launch_bounds__(1024) norms_sum_kernel(const double *__restrict__ partials, unsigned n, double *__restrict__ out)
{
   __shared__ double sh[32];
   double a = 0., b = 0.;
   for (unsigned i = threadIdx.x; i < n; i += 1024) a += partials[i], b += partials[(size_t)n + i];
   const double ta = block_sum<1024>(a, sh), tb = block_sum<1024>(b, sh);
   if (threadIdx.x == 0) out[0] = ta, out[1] = tb;
}

// ---- (|K|_F^2, trace K) of the CONSTRAINED matrix from the fused sums of the unconstrained one ----
// One warp per constrained node I, before dirichlet_kernel changes the values: sums v^2 over the
// entries that will be overwritten (rows of the constrained dofs of I, and their columns in the rows
// of dofs that are not constrained themselves: every entry once) and the diagonal entries that will
// become `diag`; norms_fix_finish_kernel then corrects the fused sums in a fixed order.
__global__ void norms_fix_kernel(int nbc, const int32_t *__restrict__ bc_nodes, const uint8_t *__restrict__ bc,
                                 const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                                 const double *__restrict__ values, double *__restrict__ partials)
{
   const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
   if (w >= nbc) return;
   const int64_t I = bc_nodes[w];
   const bool m0 = bc[2 * I], m1 = bc[2 * I + 1];
   const int64_t bi = brp[I];
   const int deg = (int)(brp[I + 1] - bi);
   const double *row0 = values + 4 * bi, *row1 = row0 + 2 * deg;
   double s2 = 0., sd = 0., cnt = 0.;
   for (int s = lane; s < deg; s += 32)
   {
      const int64_t J = bcol[bi + s];
      if (m0) s2 += row0[2 * s] * row0[2 * s] + row0[2 * s + 1] * row0[2 * s + 1];
      if (m1) s2 += row1[2 * s] * row1[2 * s] + row1[2 * s + 1] * row1[2 * s + 1];
      if (J == I)
      {
         if (m0) sd += row0[2 * s], cnt += 1.;
         if (m1) sd += row1[2 * s + 1], cnt += 1.;
         // the unconstrained dof of a half-constrained node: its entry in the constrained column
         if (m0 && !m1) s2 += row1[2 * s] * row1[2 * s];
         if (m1 && !m0) s2 += row0[2 * s + 1] * row0[2 * s + 1];
         continue;
      }
      // column I of row J (the pattern is symmetric): rows of J that are not constrained themselves
      const bool j0 = bc[2 * J], j1 = bc[2 * J + 1];
      const int64_t bj = brp[J];
      const int degj = (int)(brp[J + 1] - bj);
      int lo = 0, hi = degj;
      while (lo < hi)
      {
         const int mid = (lo + hi) >> 1;
         if (bcol[bj + mid] < I)
            lo = mid + 1;
         else
            hi = mid;
      }
      if (lo < degj && bcol[bj + lo] == I)
      {
         const double *c0 = values + 4 * bj, *c1 = c0 + 2 * degj;
         if (m0)
         {
            if (!j0) s2 += c0[2 * lo] * c0[2 * lo];
            if (!j1) s2 += c1[2 * lo] * c1[2 * lo];
         }
         if (m1)
         {
            if (!j0) s2 += c0[2 * lo + 1] * c0[2 * lo + 1];
            if (!j1) s2 += c1[2 * lo + 1] * c1[2 * lo + 1];
         }
      }
   }
   s2 = warp_sum(s2), sd = warp_sum(sd), cnt = warp_sum(cnt);
   if (lane == 0) partials[3 * w] = s2, partials[3 * w + 1] = sd, partials[3 * w + 2] = cnt;
}

__global__ void __launch_bounds__(256)
norms_fix_finish_kernel(int nbc, const double *__restrict__ partials, double diag, double *__restrict__ out)
{
   __shared__ double sh[8];
   double s2 = 0., sd = 0., cnt = 0.;
   for (int k = threadIdx.x; k < nbc; k += 256) s2 += partials[3 * k], sd += partials[3 * k + 1], cnt += partials[3 * k + 2];
   const double t2 = block_sum<256>(s2, sh), td = block_sum<256>(sd, sh), tc = block_sum<256>(cnt, sh);
   if (threadIdx.x == 0)
   {
      out[0] += tc * diag * diag - t2;
      out[1] += tc * diag - td;
   }
}

// ---- generic path: per-quadrature-point loop, damaged tangent, any family -------
template <int ET>
__device__ inline void visit_generic(const AsmArgs &A, const Visit &r, double (*kb)[4])
{
   constexpr int nd = Elem<ET>::nd, nv = Elem<ET>::nv, nq = Elem<ET>::nq;
   const int a = r.a;
   const int64_t e = r.e;
   double xv[nv][2], dv[nv];
#pragma unroll
   for (int v = 0; v < nv; ++v)
   {
      const int64_t g = A.xdofmap[e * nv + v];
      xv[v][0] = A.x[g * A.xs];
      xv[v][1] = A.x[g * A.xs + 1];
      dv[v] = A.dnod ? A.dnod[g] : 0.;
   }
   const double Ee = A.E[e];
   const double lam = Ee * A.lc.c2, mu = Ee * A.lc.c3;
#pragma unroll
   for (int b = 0; b < nd; ++b) kb[b][0] = kb[b][1] = kb[b][2] = kb[b][3] = 0.;
#pragma unroll 1
   for (int q = 0; q < nq; ++q)
   {
      double G[nd][2], phi[nv], D[9];
      const double w = qp_geometry<ET>(xv, q, G, phi);
      double d = 0.;
#pragma unroll
      for (int v = 0; v < nv; ++v) d += phi[v] * dv[v];
      if (d > 0.)
      {
         double g00 = 0., g01 = 0., g10 = 0., g11 = 0.;
         if (A.u)
#pragma unroll
            for (int b = 0; b < nd; ++b)
            {
               const int64_t gd = 2 * (int64_t)A.dofmap[e * nd + b];
               const double ux = A.u[gd], uy = A.u[gd + 1];
               g00 += ux * G[b][0];
               g01 += ux * G[b][1];
               g10 += uy * G[b][0];
               g11 += uy * G[b][1];
            }
         const double s = 0.5 * (g01 + g10);
         const double eps[4] = {g00, s, s, g11};
         tangent(A.variant, lam, mu, d, eps, D);
      }
      else
         hooke_scaled(lam, mu, 1., D);
      double ga[2] = {0., 0.};
#pragma unroll
      for (int b = 0; b < nd; ++b)
         if (b == a) ga[0] = G[b][0], ga[1] = G[b][1];
#pragma unroll
      for (int b = 0; b < nd; ++b) bdb_block(ga, G[b], D, w, kb[b]);
   }
}

// One thread owns one block row (node I) of a tile of R consecutive node rows and
// walks the cells incident to I.  Threads are assigned to nodes in order of
// DECREASING visit count (P2: vertex nodes have 6 incident cells, edge nodes 2), so
// the lanes of a warp run the same number of visits; on the fast path the three
// dependent load levels are issued for CH visits at a time.
template <int ET, bool FAST, int CH, int TPN, bool DMG>
__global__ void __launch_bounds__(kAsmR * TPN) assemble_kernel(AsmArgs A)
{
   constexpr int nd = Elem<ET>::nd, R = kAsmR, THREADS = kAsmR * TPN;
   extern __shared__ double2 sv[];
   // fast path: two threads per node (one per scalar row); generic path: one
   const int tid = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * R;
   const int nloc = (int)min((int64_t)R, A.nnodes - n0);
   const int64_t b0 = A.brp[n0];
   const int32_t vbase = A.nptr[n0];
   const int units = 2 * (int)(A.brp[n0 + nloc] - b0);  // 16-byte units of this tile
   // tile metadata behind the staging area
   int32_t *s_cnt = reinterpret_cast<int32_t *>(sv + A.stage_units);  // number of visits of node i
   int32_t *s_roff = s_cnt + R;                                        // unit offset of row 0, [R + 1]
   int32_t *s_voff = s_roff + R + 1;                                   // [kAsmLevels] level offsets of the records
   if (tid < nloc)
   {
      s_cnt[tid] = A.nptr[n0 + tid + 1] - A.nptr[n0 + tid];
      s_roff[tid] = 2 * (int)(A.brp[n0 + tid] - b0);
   }
   if (tid == 0) s_roff[nloc] = units;
   if (tid < kAsmLevels) s_voff[tid] = A.voff[(int64_t)blockIdx.x * kAsmLevels + tid];
   // TPN == 2: lanes 0-15 of a warp own scalar row 0 of 16 nodes, lanes 16-31 row 1 of the same
   // nodes: the 8 lanes of a shared-memory phase then belong to 8 different nodes.  Ranks are the
   // plan's order of decreasing visit count: the lanes of a warp run the same number of visits.
   const int rank = TPN == 2 ? ((tid >> 5) << 4) + (tid & 15) : tid;
   const int half = TPN == 2 ? ((tid >> 4) & 1) : 0;
   const int i = rank < nloc ? (int)A.perm[n0 + rank] : 0;
   __syncthreads();
   if (rank < nloc)
   {
      const int cnt = s_cnt[i];
      const int r0 = s_roff[i];
      const int r1 = r0 + ((s_roff[i + 1] - r0) >> 1);
      const uint4 *rec = reinterpret_cast<const uint4 *>(A.vrec + vbase) + rank;
      if (FAST)
      {
         // software pipeline over the visits: while batch c is computed and staged, the cell records
         // of batch c + CH and the visit records of batch c + 2 CH are in flight
         uint4 raw[CH], raw1[CH], raw2[CH];
         FastGeo geo[CH], geo1[CH];
         const uint4 none = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
         for (int j = 0; j < CH; ++j) raw1[j] = (j < cnt) ? rec[s_voff[j]] : none;
#pragma unroll
         for (int j = 0; j < CH; ++j) raw2[j] = (CH + j < cnt) ? rec[s_voff[CH + j]] : none;
#pragma unroll
         for (int j = 0; j < CH; ++j)
            if (j < cnt) geo1[j] = fast_geo(A, Visit(raw1[j]));
         for (int c = 0; c < cnt; c += CH)
         {
#pragma unroll
            for (int j = 0; j < CH; ++j) raw[j] = raw1[j], geo[j] = geo1[j], raw1[j] = raw2[j];
#pragma unroll
            for (int j = 0; j < CH; ++j)
               if (c + CH + j < cnt) geo1[j] = fast_geo(A, Visit(raw1[j]));
#pragma unroll
            for (int j = 0; j < CH; ++j) raw2[j] = (c + 2 * CH + j < cnt) ? rec[s_voff[c + 2 * CH + j]] : none;
#pragma unroll
            for (int j = 0; j < CH; ++j)
               if (c + j < cnt)
               {
                  if (DMG && geo[j].g1x != geo[j].g1x)
                  {  // damaged cell: NaN marker, its damage record is celld[cell]
                     if (TPN == 2)
                        damaged_compute_stage<ET>(A, Visit(raw[j]), sv, half ? r1 : r0, half);
                     else
                     {
                        damaged_compute_stage<ET>(A, Visit(raw[j]), sv, r0, 0);
                        damaged_compute_stage<ET>(A, Visit(raw[j]), sv, r1, 1);
                     }
                  }
                  else if (TPN == 2)
                     fast_compute_stage<ET>(A, Visit(raw[j]), geo[j], sv, half ? r1 : r0, half);
                  else
                  {
                     fast_compute_stage<ET>(A, Visit(raw[j]), geo[j], sv, r0, 0);
                     fast_compute_stage<ET>(A, Visit(raw[j]), geo[j], sv, r1, 1);
                  }
               }
         }
      }
      else
      {
         for (int c = 0; c < cnt; ++c)
         {
            const Visit r(rec[s_voff[c]]);
            double kb[nd][4];
            visit_generic<ET>(A, r, kb);
#pragma unroll
            for (int b = 0; b < nd; ++b)
            {
               const int t = stored_position(b, (int)r.a, nd);
               stage_block(sv, r0, r1, r.slot(t), kb[b], r.is_first(t));
            }
         }
      }
   }
   __syncthreads();
   // stream the finished tile out: one contiguous byte range of the CSR values
   double *dst = A.values + 4 * b0;
   const int padded = (units + 7) & ~7;
   for (int k = tid; k < padded; k += THREADS)
   {
      const int u = swz(k);
      if (u < units) st_stream_d2(dst + 2 * (int64_t)u, sv[k]);
   }
}

// ---- Dirichlet rows / columns / diagonal (F.cc:852-857) --------------------------
// one warp per constrained node I; lanes over the blocks of row I.  Zeroing summed
// values equals summing zeroed element contributions exactly, so this matches the
// element-level treatment of dolfinx bit for bit.
__global__ void dirichlet_kernel(int nbc, const int32_t *__restrict__ bc_nodes, const uint8_t *__restrict__ bc,
                                 const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                                 double *__restrict__ values, double diag)
{
   const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
   if (w >= nbc) return;
   const int64_t I = bc_nodes[w];
   const bool m0 = bc[2 * I], m1 = bc[2 * I + 1];
   const int64_t bi = brp[I];
   const int deg = (int)(brp[I + 1] - bi);
   double *row0 = values + 4 * bi, *row1 = row0 + 2 * deg;
   int self = -1;
   for (int s = lane; s < deg; s += 32)
   {
      const int64_t J = bcol[bi + s];
      if (J == I) self = s;
      if (m0) row0[2 * s] = row0[2 * s + 1] = 0.;
      if (m1) row1[2 * s] = row1[2 * s + 1] = 0.;
      // column I of row J (the pattern is symmetric)
      const int64_t bj = brp[J];
      const int degj = (int)(brp[J + 1] - bj);
      int lo = 0, hi = degj;
      while (lo < hi)
      {
         const int mid = (lo + hi) >> 1;
         if (bcol[bj + mid] < I)
            lo = mid + 1;
         else
            hi = mid;
      }
      if (lo < degj && bcol[bj + lo] == I)
      {
         double *c0 = values + 4 * bj, *c1 = c0 + 2 * degj;
         if (m0) c0[2 * lo] = c1[2 * lo] = 0.;
         if (m1) c0[2 * lo + 1] = c1[2 * lo + 1] = 0.;
      }
   }
   __syncwarp();
   if (self >= 0)
   {  // set_diagonal(..., diag) with INSERT_VALUES (F.cc:857)
      if (m0) row0[2 * self] = diag;
      if (m1) row1[2 * self + 1] = diag;
   }
}

// ---- Frobenius norm^2 and trace --------------------------------------------------
// fro^2: one flat streaming pass over the value array; trace: one thread per node looks its
// diagonal block up in the (sorted) block row.  Deterministic reductions.
__global__ void __launch_bounds__(256)
fro_kernel(int64_t n2, const double2 *__restrict__ values, ReduceScratch red, double *__restrict__ out)
{
   double acc = 0.;
   const int64_t stride = (int64_t)gridDim.x * 256;
   for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n2; i += stride)
   {
      const double2 v = ld_stream_d2(reinterpret_cast<const double *>(values + i));
      acc += v.x * v.x + v.y * v.y;
   }
   block_reduce_finish<256>(acc, red, out);
}

__global__ void __launch_bounds__(256)
trace_kernel(int64_t nnodes, const int64_t *__restrict__ brp, const uint8_t *__restrict__ dslot,
             const double *__restrict__ values, ReduceScratch red, double *__restrict__ out)
{
   double acc = 0.;
   const int64_t stride = (int64_t)gridDim.x * 256;
   for (int64_t I = (int64_t)blockIdx.x * 256 + threadIdx.x; I < nnodes; I += stride)
   {
      const int64_t bi = brp[I];
      const int deg = (int)(brp[I + 1] - bi), s = dslot[I];
      if (s < deg) acc += values[4 * bi + 2 * s] + values[4 * bi + 2 * deg + 2 * s + 1];
   }
   block_reduce_finish<256>(acc, red, out);
}

template <int ET, bool FAST, int CH, int TPN, bool DMG = false>
static int launch_assemble_ch(const femb200_plan *p, AsmArgs A, cudaStream_t st)
{
   static_assert(tile_r(1) == kAsmR, "tile_max_blocks[1] must describe kAsmR-row tiles");
   const size_t budget = devinfo().smem_optin ? devinfo().smem_optin : 227 * 1024;
   A.stage_units = (2 * p->tile_max_blocks[1] + 7) & ~7;
   const size_t smem = 16 * (size_t)A.stage_units + 4 * (size_t)(2 * kAsmR + 1 + kAsmLevels) + 16;
   FEMB_CHECK(smem <= budget, "assemble: a %d-node tile needs %zu B of shared memory (> %zu)", kAsmR, smem, budget);
   if (int rc = ensure_dynamic_smem<assemble_kernel<ET, FAST, CH, TPN, DMG>>(smem)) return rc;
   const unsigned grid = (unsigned)cdiv(p->nnodes, kAsmR);
   assemble_kernel<ET, FAST, CH, TPN, DMG><<<grid, kAsmR * TPN, smem, st>>>(A);
   FEMB_LAUNCH_CHECK();
   return 0;
}

template <int ET, bool DMG, bool NORMS, int MINB, bool STAGE>
static int launch_fast_kernel(const femb200_plan *p, AsmArgs A, const ReduceScratch &red, double *d_norms, cudaStream_t st)
{
   femb200_plan *pm = const_cast<femb200_plan *>(p);
   const size_t smem = 16 * (size_t)A.stage_units + (STAGE ? kDmgStageBytes + 16 + 4 * dmg_stage_cap<ET>() : 0);
   const unsigned grid = (unsigned)cdiv(p->nnodes, kAsmR);
   const CUtensorMap &tm8 = *reinterpret_cast<const CUtensorMap *>(pm->tmap[0]), &tm1 = *reinterpret_cast<const CUtensorMap *>(pm->tmap[1]);
   if (int rc = ensure_dynamic_smem<assemble_fast_kernel<ET, DMG, NORMS, MINB, STAGE>>(smem)) return rc;
   assemble_fast_kernel<ET, DMG, NORMS, MINB, STAGE><<<grid, kAsmR * 2, smem, st>>>(A, red, d_norms, tm8, tm1);
   FEMB_LAUNCH_CHECK();
   return 0;
}

// DMG: with A.tdam (the pre-pass wrote the tiles' rows of damaged cells) the variant that stages the damage records in
// shared memory (P2: 55 KB per CTA, compiled for the 4 CTAs per SM that fit; P1: 40 KB, 5 CTAs), else the variant whose
// visits read the records from global memory (5 CTAs per SM): faster while few cells are damaged.  assemble_matrix_impl
// chooses.
template <int ET, bool DMG, bool NORMS>
static int launch_assemble_fast_n(const femb200_plan *p, AsmArgs A, cudaStream_t st, double *d_norms)
{
   // the image starts at the tile's offset inside its 128-byte line (up to 6 units) and is whole lines
   A.stage_units = (2 * p->tile_max_blocks[1] + 6 + 7) & ~7;
   A.flevels = p->flevels;
   A.prefetch_tiles = p->opt_prefetch_tiles >= 0 ? p->opt_prefetch_tiles : 8 * devinfo().sm_count;  // a good wave of resident CTAs ahead
   const unsigned grid = (unsigned)cdiv(p->nnodes, kAsmR);
   femb200_plan *pm = const_cast<femb200_plan *>(p);
   A.use_tma = (!NORMS && p->opt_stream_out == 0 && values_tensor_maps(pm, A.values)) ? 1 : 0;
   ReduceScratch red{nullptr, nullptr};
   if (NORMS)
      if (int rc = reduce_scratch(grid, st, &red, 2)) return rc;
   int rc;
   if (DMG && A.tdam)
      rc = launch_fast_kernel<ET, DMG, NORMS, DMG ? (ET == FEMB200_P1 ? 5 : 4) : 7, DMG>(p, A, red, d_norms, st);
   else
      rc = launch_fast_kernel<ET, DMG, NORMS, DMG ? 5 : (ET == FEMB200_P1 ? 8 : 7), false>(p, A, red, d_norms, st);
   if (rc) return rc;
   if (NORMS)
   {
      norms_sum_kernel<<<1, 1024, 0, st>>>(red.partials, grid, d_norms);
      FEMB_LAUNCH_CHECK();
   }
   return 0;
}

template <int ET, bool DMG>
static int launch_assemble_fast(const femb200_plan *p, AsmArgs A, cudaStream_t st, double *d_norms)
{
   return d_norms ? launch_assemble_fast_n<ET, DMG, true>(p, A, st, d_norms) : launch_assemble_fast_n<ET, DMG, false>(p, A, st, d_norms);
}

// *fused: in: the caller wants (|K|_F^2, trace K) in d_norms; out: whether the kernel produced them
template <int ET, bool FAST>
static int launch_assemble(const femb200_plan *p, const AsmArgs &A, cudaStream_t st, double *d_norms, bool *fused)
{
   *fused = false;
   if (!FAST) return launch_assemble_ch<ET, FAST, 1, 1>(p, A, st);
   if (ET != FEMB200_Q2 && A.frec && p->opt_assembly_path != 1)
   {
      constexpr int TRI = ET == FEMB200_Q2 ? FEMB200_P2 : ET;
      *fused = d_norms != nullptr;
      return A.celld ? launch_assemble_fast<TRI, true>(p, A, st, d_norms) : launch_assemble_fast<TRI, false>(p, A, st, d_norms);
   }
   // older record format (16-byte visit records, staging addresses computed per block): plans without
   // fast records (a node in 16 cells, a staging image over 32 KB) and plans with assembly_path = 1
   if (A.celld) return launch_assemble_ch<ET, FAST, 1, 2, true>(p, A, st);  // damaged cells present
   return launch_assemble_ch<ET, FAST, 1, 2>(p, A, st);
}

}  // namespace femb

using namespace femb;

static int assemble_matrix_impl(const femb200_plan *p, const double *d_x, int x_stride, const double *d_E, double nu,
                                const double *d_dnod, const double *d_u, int variant, double *d_values, void *stream,
                                bool dirichlet, double *d_norms = nullptr)
{
   FEMB_CHECK(p && d_x && d_E && d_values, "assemble_matrix: null argument");
   FEMB_REFUSE_Q1(p->etype, "assemble_matrix");
   FEMB_CHECK(x_stride == 2 || x_stride == 3, "assemble_matrix: x_stride must be 2 or 3, got %d", x_stride);
   AsmArgs A;
   A.nnodes = p->nnodes, A.nptr = p->nptr, A.vrec = p->vrec, A.frec = p->frec, A.tcnt = p->tcnt, A.thdr = p->thdr, A.perm = p->perm, A.voff = p->voff, A.brp = p->brp;
   A.xdofmap = p->xdofmap, A.dofmap = p->dofmap, A.x = d_x, A.xs = x_stride, A.E = d_E, A.lc = lame_coef(nu);
   A.dnod = d_dnod, A.u = d_u, A.variant = variant, A.values = d_values;
   cudaStream_t st = as_stream(stream);
   // triangles take the per-cell pre-pass + fast kernel (damaged cells through their own per-cell
   // tangent records); Q2 and plans with assembly_path = 2 take the per-quadrature-point kernel
   const bool linear = (p->etype != FEMB200_Q2) && p->opt_assembly_path != 2;
   A.cellrec = nullptr, A.celld = nullptr, A.tdam = nullptr;
   if (linear)
   {
      femb200_plan *pm = const_cast<femb200_plan *>(p);  // lazily allocated scratch of the plan
      if (!pm->cellrec)
      {
         std::lock_guard<std::mutex> lock(pm->range_mtx);
         if (!pm->cellrec)
         {
            FEMB_CUDA(cudaMalloc(&pm->cellrec, sizeof(double) * 4 * (size_t)p->ncells));
            pm->bytes += sizeof(double) * 4 * (size_t)p->ncells;
         }
      }
      const unsigned grid = (unsigned)cdiv(p->ncells, 128);
      if (d_dnod)
      {
         // one damage record per cell at worst (192-byte slots for P2): the plan's per-cell scratch, allocated on first use
         static_assert(dmg_rec_doubles<FEMB200_P1>() == 12 && dmg_rec_doubles<FEMB200_P2>() == 24, "plan_cell_scratch_doubles");
         if (int rc = plan_cell_scratch(pm)) return rc;
         // The fast kernel can stage the damage records of a tile's cells in shared memory (slot map of the plan, built
         // when first needed, + the per-assembly rows of damaged cells the pre-pass writes through it): that wins once
         // about 40 % of the cells are damaged (n = 1448: 1.56 against 1.65 ms at 50 %, 1.89 against 2.39 ms at 100 %)
         // and loses below (1.30 against 1.09 ms at 10 %: 4 CTAs per SM instead of 5).  The choice follows the share
         // of damaged cells of the PREVIOUS damaged assembly on this plan, which the pre-pass leaves in host-mapped
         // memory (read here without synchronisation): it affects speed only, both kernels assemble the same matrix.
         const bool fastk = p->frec && p->opt_assembly_path != 1;
         const int cap = p->etype == FEMB200_P1 ? dmg_stage_cap<FEMB200_P1>() : dmg_stage_cap<FEMB200_P2>();
         if (!pm->dmg_count)
         {
            std::lock_guard<std::mutex> lock(pm->range_mtx);
            if (!pm->dmg_count)
            {
               int *h = nullptr;
               FEMB_CUDA(cudaHostAlloc(&h, sizeof(int), cudaHostAllocMapped));
               *h = 0;
               FEMB_CUDA(cudaHostGetDevicePointer(&pm->dmg_count_dev, h, 0));
               FEMB_CUDA(cudaMalloc(&pm->dmg_counter, sizeof(int)));
               FEMB_CUDA(cudaMemset(pm->dmg_counter, 0, sizeof(int)));
               pm->dmg_count = h;
            }
         }
         const int64_t last = *static_cast<volatile int *>(pm->dmg_count);
         const bool staged = fastk && (p->opt_dmg_stage == 1 || (p->opt_dmg_stage == 0 && last * 5 >= p->ncells * 2));
         if (staged)
            if (int rc = plan_tile_cells(pm, cap, st)) return rc;
         const uint4 *cref = (staged && pm->tdam_refs) ? reinterpret_cast<const uint4 *>(pm->cref) : nullptr;
         const int spec = last * 5 >= p->ncells * 2;  // most cells damaged last time: the pre-pass gathers u before it tests d
         if (p->etype == FEMB200_P1)
            cell_setup_damage_kernel<FEMB200_P1><<<grid, 128, 0, st>>>(p->ncells, p->xdofmap, p->dofmap, d_x, x_stride, d_E, A.lc,
                                                                       d_dnod, d_u, variant, pm->cellrec, pm->celld, cref, pm->tdam, cap,
                                                                       pm->dmg_counter, spec);
         else
            cell_setup_damage_kernel<FEMB200_P2><<<grid, 128, 0, st>>>(p->ncells, p->xdofmap, p->dofmap, d_x, x_stride, d_E, A.lc,
                                                                       d_dnod, d_u, variant, pm->cellrec, pm->celld, cref, pm->tdam, cap,
                                                                       pm->dmg_counter, spec);
         dmg_count_publish_kernel<<<1, 1, 0, st>>>(pm->dmg_counter, pm->dmg_count_dev);
         A.tdam = staged ? pm->tdam : nullptr;
         A.celld = pm->celld;
      }
      else
         cell_setup_kernel<<<(unsigned)cdiv(p->ncells, 256), 256, 0, st>>>(p->ncells, p->xdofmap, d_x, x_stride, d_E,
                                                                           A.lc, pm->cellrec);
      FEMB_LAUNCH_CHECK();
      A.cellrec = pm->cellrec;
   }
   int rc;
   bool fused = false;
   switch (p->etype)
   {
      case FEMB200_P1:
         rc = linear ? launch_assemble<FEMB200_P1, true>(p, A, st, d_norms, &fused)
                     : launch_assemble<FEMB200_P1, false>(p, A, st, d_norms, &fused);
         break;
      case FEMB200_P2:
         rc = linear ? launch_assemble<FEMB200_P2, true>(p, A, st, d_norms, &fused)
                     : launch_assemble<FEMB200_P2, false>(p, A, st, d_norms, &fused);
         break;
      default:
         rc = launch_assemble<FEMB200_Q2, false>(p, A, st, d_norms, &fused);
   }
   if (rc) return rc;
   const bool constrained = dirichlet && p->bc && p->nbc > 0;
   if (d_norms && fused && constrained)
   {  // correct the fused sums of the unconstrained matrix for the entries the Dirichlet kernel overwrites
      femb200_plan *pm = const_cast<femb200_plan *>(p);
      if (!pm->norm_partials)
      {
         FEMB_CUDA(cudaMalloc(&pm->norm_partials, sizeof(double) * 3 * (size_t)p->nbc));
         pm->bytes += sizeof(double) * 3 * (size_t)p->nbc;
      }
      norms_fix_kernel<<<(unsigned)cdiv((int64_t)p->nbc * 32, 128), 128, 0, st>>>(p->nbc, p->bc_nodes, p->bc, p->brp, p->bcol,
                                                                                  d_values, pm->norm_partials);
      norms_fix_finish_kernel<<<1, 256, 0, st>>>(p->nbc, pm->norm_partials, 1.0, d_norms);
      FEMB_LAUNCH_CHECK();
   }
   if (constrained)
      if (int rc2 = femb200_apply_dirichlet(p, d_values, 1.0, stream)) return rc2;
   if (d_norms && !fused) return femb200_matrix_norms(p, d_values, d_norms, stream);  // other kernels: separate pass
   return 0;
}

extern "C" int femb200_assemble_matrix(const femb200_plan *p, const double *d_x, int x_stride, const double *d_E,
                                       double nu, const double *d_dnod, const double *d_u, int variant,
                                       double *d_values, void *stream)
{
   return assemble_matrix_impl(p, d_x, x_stride, d_E, nu, d_dnod, d_u, variant, d_values, stream, true);
}

extern "C" int femb200_assemble_matrix_norms(const femb200_plan *p, const double *d_x, int x_stride, const double *d_E,
                                             double nu, const double *d_dnod, const double *d_u, int variant,
                                             double *d_values, double *d_norms, void *stream)
{
   FEMB_CHECK(d_norms != nullptr, "assemble_matrix_norms: null output");
   return assemble_matrix_impl(p, d_x, x_stride, d_E, nu, d_dnod, d_u, variant, d_values, stream, true, d_norms);
}

extern "C" int femb200_assemble_matrix_nobc(const femb200_plan *p, const double *d_x, int x_stride, const double *d_E,
                                            double nu, const double *d_dnod, const double *d_u, int variant,
                                            double *d_values, void *stream)
{
   return assemble_matrix_impl(p, d_x, x_stride, d_E, nu, d_dnod, d_u, variant, d_values, stream, false);
}

extern "C" int femb200_apply_dirichlet(const femb200_plan *p, double *d_values, double diag, void *stream)
{
   FEMB_CHECK(p && d_values, "apply_dirichlet: null argument");
   if (!p->bc || p->nbc == 0) return 0;
   const int T = 128;
   dirichlet_kernel<<<(unsigned)cdiv((int64_t)p->nbc * 32, T), T, 0, as_stream(stream)>>>(
       p->nbc, p->bc_nodes, p->bc, p->brp, p->bcol, d_values, diag);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_matrix_norms(const femb200_plan *p, const double *d_values, double *d_out, void *stream)
{
   FEMB_CHECK(p && d_values && d_out, "matrix_norms: null argument");
   cudaStream_t st = as_stream(stream);
   const int64_t n2 = 2 * p->nnzb;  // 16-byte units of the value array
   const unsigned g1 = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(n2, 256), (int64_t)devinfo().sm_count * 16));
   const unsigned g2 = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(p->nnodes, 256), (int64_t)devinfo().sm_count * 16));
   ReduceScratch red;
   if (int rc = reduce_scratch(std::max(g1, g2), st, &red)) return rc;
   fro_kernel<<<g1, 256, 0, st>>>(n2, reinterpret_cast<const double2 *>(d_values), red, d_out);
   FEMB_LAUNCH_CHECK();
   trace_kernel<<<g2, 256, 0, st>>>(p->nnodes, p->brp, p->dslot, d_values, red, d_out + 1);
   FEMB_LAUNCH_CHECK();
   return 0;
}
