// spmv.cu -- assembled operator apply y = A x on the node-block pattern.
//
// Role in the reference: HypreParMatrix::Mult inside mfem::CGSolver
// (M.cc:1502,1525-1528) / PETSc MatMult inside KSP cg (F.cc:718-722).
//
// The matrix values live in the scalar-CSR layout handed across the boundary
// (row 2I: 2 deg doubles, row 2I+1: 2 deg doubles, contiguous), but the kernel
// walks the node-block pattern (brp/bcol): one int32 column index per 2x2 block
// instead of four, i.e. 36 B per block instead of 48 B.  Eight lanes own one
// node row pair; lane s handles blocks s, s+8, ...: 16-byte loads of both
// scalar rows and of x[2J..2J+1], shuffle reduction over the eight lanes.
// <x, y> is optionally fused (CG needs <d, A d>): deterministic two-stage
// reduction (block partials, last block sums them in a fixed order).
#include <algorithm>
#include <mutex>
#include <type_traits>

#include "plan.cuh"
#include "reduce.cuh"
#include "tma.cuh"

namespace femb {

constexpr int kSpmvLanes = 8;
constexpr int kSpmvThreads = 256;

template <bool DOT>
__global__ void __launch_bounds__(kSpmvThreads)
spmv_kernel(int64_t row_lo, int64_t nnodes, const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
            const double *__restrict__ values, const double *__restrict__ x, double *__restrict__ y,
            const double *__restrict__ flag, ReduceScratch red, double *__restrict__ out, bool accumulate = false)
{
   if (flag && *flag != 0.) return;  // converged CG: become a no-op (uniform over the grid)
   const int lane = threadIdx.x & (kSpmvLanes - 1);
   const int64_t I = row_lo + ((int64_t)blockIdx.x * kSpmvThreads + threadIdx.x) / kSpmvLanes;
   double y0 = 0., y1 = 0.;
   if (I < nnodes)
   {
      const int64_t bi = brp[I];
      const int deg = (int)(brp[I + 1] - bi);
      const double2 *row0 = reinterpret_cast<const double2 *>(values + 4 * bi);
      const double2 *row1 = row0 + deg;
      const int32_t *cols = bcol + bi;
      const double2 *x2 = reinterpret_cast<const double2 *>(x);
      // three blocks per lane in flight (deg <= 24 covers P1/P2/Q2 interior rows)
      int s = lane;
      for (; s + 2 * kSpmvLanes < deg; s += 3 * kSpmvLanes)
      {
         const int32_t j0 = cols[s], j1 = cols[s + kSpmvLanes], j2 = cols[s + 2 * kSpmvLanes];
         const double2 a0 = row0[s], a1 = row0[s + kSpmvLanes], a2 = row0[s + 2 * kSpmvLanes];
         const double2 c0 = row1[s], c1 = row1[s + kSpmvLanes], c2 = row1[s + 2 * kSpmvLanes];
         const double2 v0 = x2[j0], v1 = x2[j1], v2 = x2[j2];
         y0 += a0.x * v0.x + a0.y * v0.y + a1.x * v1.x + a1.y * v1.y + a2.x * v2.x + a2.y * v2.y;
         y1 += c0.x * v0.x + c0.y * v0.y + c1.x * v1.x + c1.y * v1.y + c2.x * v2.x + c2.y * v2.y;
      }
      for (; s < deg; s += kSpmvLanes)
      {
         const int32_t j0 = cols[s];
         const double2 a0 = row0[s], c0 = row1[s], v0 = x2[j0];
         y0 += a0.x * v0.x + a0.y * v0.y;
         y1 += c0.x * v0.x + c0.y * v0.y;
      }
   }
#pragma unroll
   for (int o = kSpmvLanes / 2; o > 0; o >>= 1)
   {
      y0 += __shfl_xor_sync(0xffffffffu, y0, o);
      y1 += __shfl_xor_sync(0xffffffffu, y1, o);
   }
   double part = 0.;
   if (I < nnodes && lane == 0)
   {
      reinterpret_cast<double2 *>(y)[I] = make_double2(y0, y1);
      if (DOT)
      {
         const double2 xi = reinterpret_cast<const double2 *>(x)[I];
         part = xi.x * y0 + xi.y * y1;
      }
   }
   if (DOT) block_reduce_finish<kSpmvThreads>(part, red, out, accumulate);
}

// ---------------------------------------------------------------------------
// TMA-staged persistent variant (default).  The node rows [n0, n0 + R) of a tile
// own one contiguous byte range of the value array, of bcol and of brp: a producer
// warp streams those ranges into shared memory with 1-D bulk copies
// (cp.async.bulk -> UBLKCP) completing on an mbarrier, S stages deep, while eight
// consumer warps (L lanes per node row pair) reduce the previous tiles out of shared memory; the only
// per-thread global loads left are the gathers of x (L1/L2 hits: the lattice
// numbering keeps the reuse window at a few node rows).  Grid = resident CTAs only,
// so the fused <x, y> needs ~300 tickets instead of one per 32 rows.
// ---------------------------------------------------------------------------
constexpr int kTmaConsumers = 256;
constexpr int kTmaThreads = kTmaConsumers + 32;

struct SpmvTile
{
   int vbytes, cbytes, pbytes;  // stage capacities: values, column indices (or stencil ids), row pointers
};

// Column modes.  C32: the plan's bcol.  C16: its 16-bit offsets from the row's own node (bcol16: every |J - I| of the
// pattern fits, which any numbering with locality gives: the lattice numbering of config 4 has |J - I| <= 2 (2 n + 1) + 2
// = 23 172): 34 instead of 36 bytes per node block.  STENCIL: one byte per node row, the row's id in the plan's stencil
// dictionary (the distinct bcol16 lists: 16 on a P2 lattice), which the CTA holds in shared memory: 32 bytes per node
// block and one per node row, no column indices and no brp stage.  The producer warp reads a tile's ids two tiles
// ahead, turns them into value offsets (warp scan over the dictionary degrees) one tile ahead, and stores one word per
// row, (offset | id << 16), into the stage next to the values before it arrives on the stage's barrier: the consumers'
// dependent chain stays as short as with brp, and no global read sits between a free stage and its value copy (with
// the scan in the consumers the apply was 4 % slower than the 16-bit mode).  All three modes apply the same products in
// the same order: y and <x, y> agree bit for bit.
// Two more modes serve the PCG (cg.cu) on plans with compact values (plan.cuh): kCompactWrite streams the CSR values like
// kStencil, with rows described by their compact keys, and also writes every kept block into p->cvalues and checks that
// every dropped block is +-0 (else *cbad = 1).  kCompact streams the compact values (about 3/4 of the bytes on a P2
// mesh): a dropped slot takes +0 for its block and its x (no shared-memory read, no gather) instead of its stored +-0
// block and x, and everything else -- grid, tiles, lanes,
// the products and their order -- is the stencil mode's.  The sign of a zero product cannot reach y: a chain whose
// products are +-0 until a non-zero one has the value of that product from there on; a chain that is +-0 throughout
// adds +-0 to y0, which starts at +0 and is never -0 (x finite).  So y and <x, y> agree bit for bit.
enum SpmvCols
{
   kC32 = 0,
   kC16 = 1,
   kStencil = 2,
   kCompactWrite = 3,
   kCompact = 4
};
// shared-memory dictionary entry: kStencilD offsets, the degree, one pad entry (17 words: rows of different ids start in
// different banks)
constexpr int kDictStride = kStencilD + 2;

struct SpmvStencils
{
   const uint8_t *sig;       // [nnodes]  (compact modes: the compact keys)
   const int16_t *off;       // [k][kStencilD]  (compact modes: the entries [k][kCDictStride])
   const uint8_t *deg;       // [k]
   int k;
};

// compact values (kCompactWrite / kCompact); cbad also gates the CSR kernel that stands in for kCompact: with cbad
// non-null the other modes run only when *cbad != 0
struct SpmvCompactArgs
{
   const int64_t *cbrp;
   double *cvalues;
   int *cbad;
};

// one 2-row product chain of up to three blocks, in the order the stencil kernel has always rounded it (SASS:
// DMUL of the second product, then DFMAs of the first and of the following ones)
__device__ __forceinline__ double chain(double2 a0, double2 v0)
{
   return __fma_rn(a0.x, v0.x, __dmul_rn(a0.y, v0.y));
}
__device__ __forceinline__ double chain(double2 a0, double2 v0, double2 a1, double2 v1)
{
   return __fma_rn(a1.y, v1.y, __fma_rn(a1.x, v1.x, chain(a0, v0)));
}
__device__ __forceinline__ double chain(double2 a0, double2 v0, double2 a1, double2 v1, double2 a2, double2 v2)
{
   return __fma_rn(a2.y, v2.y, __fma_rn(a2.x, v2.x, chain(a0, v0, a1, v1)));
}

// block of slot t of a row in the stage (kCompact: at its compact position, +0 when dropped)
template <int COLS>
__device__ __forceinline__ double2 stage_block(const int16_t *cpos, const double2 *row, int t)
{
   if constexpr (COLS == kCompact)
   {
      const int c = cpos[t];
      return c >= 0 ? row[c] : make_double2(0., 0.);
   }
   else
      return row[t];
}

// x block of slot t (kCompact: +0 for a dropped slot, whose product is +-0 whatever x is when x is finite: no gather)
template <int COLS, typename col_t>
__device__ __forceinline__ double2 x_block(const int16_t *cpos, const double2 *xr, const col_t *cols, int t)
{
   if constexpr (COLS == kCompact)
   {
      if (cpos[t] < 0) return make_double2(0., 0.);
   }
   return xr[cols[t]];
}

// kCompactWrite: copies the block of slot t (rows 0 and 1) to its compact position, or checks that the dropped block is
// +-0 (a NaN is not)
template <int COLS>
__device__ __forceinline__ void put(const int16_t *cpos, double2 *cv0, double2 *cv1, int *cbad, int t, double2 a, double2 c)
{
   if constexpr (COLS == kCompactWrite)
   {
      const int k = cpos[t];
      if (k >= 0)
         cv0[k] = a, cv1[k] = c;
      else if (!(a.x == 0. && a.y == 0. && c.x == 0. && c.y == 0.))
         *cbad = 1;
   }
}

template <bool DOT, int R, int kTmaStages, int L, int COLS>
__global__ void __launch_bounds__(kTmaThreads)
spmv_tma_kernel(int64_t row_lo, int64_t row_hi, const int64_t *__restrict__ brp, const void *__restrict__ bcol_any,
                SpmvStencils dict, const double *__restrict__ values, const double *__restrict__ x, double *__restrict__ y,
                const double *__restrict__ flag, ReduceScratch red, double *__restrict__ out, SpmvTile cap, int ntiles,
                bool accumulate, SpmvCompactArgs ca)
{
   constexpr bool DICT = COLS >= kStencil;                // rows described by dictionary ids
   constexpr int DS = COLS >= kCompactWrite ? kCDictStride : kDictStride;
   static_assert(!DICT || R == 64, "the stencil scan covers 64 rows (two per lane of the producer warp)");
   extern __shared__ __align__(128) unsigned char smem[];
   __shared__ uint64_t full[kTmaStages], empty[kTmaStages];
   if (flag && *flag != 0.) return;  // converged CG: become a no-op (uniform over the grid)
   if (COLS == kCompact ? *ca.cbad != 0 : (COLS != kCompactWrite && ca.cbad && *ca.cbad == 0)) return;
   const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
   const int stage_bytes = cap.vbytes + cap.cbytes + cap.pbytes;
   int16_t *sdict = reinterpret_cast<int16_t *>(smem + (size_t)kTmaStages * stage_bytes);
   if constexpr (COLS == kStencil)  // the dictionary, once per CTA (published by the __syncthreads below)
      for (int e = tid; e < dict.k * kDictStride; e += kTmaThreads)
      {
         const int k = e / kDictStride, t = e - k * kDictStride;
         sdict[e] = t < kStencilD ? dict.off[k * kStencilD + t] : t == kStencilD ? (int16_t)dict.deg[k] : (int16_t)0;
      }
   else if constexpr (DICT)
      for (int e = tid; e < dict.k * kCDictStride; e += kTmaThreads) sdict[e] = dict.off[e];
   if (tid == 0)
   {
#pragma unroll
      for (int s = 0; s < kTmaStages; ++s)
      {
         mbar_init(&full[s], 1);
         mbar_init(&empty[s], kTmaConsumers / 32);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
   }
   __syncthreads();
   const int first = blockIdx.x, stride = gridDim.x;
   const int nmine = first < ntiles ? (ntiles - first + stride - 1) / stride : 0;
   double part = 0.;
   if (warp == kTmaConsumers / 32)
   {  // ---- producer warp: one lane issues the bulk copies ----
      if constexpr (DICT)
      {  // the whole warp; lane l resolves rows 2 l and 2 l + 1.  What a tile needs besides its stage is prepared ahead
         // while the consumers still hold the stages: the global reads (first node block, ids) two tiles ahead, the
         // value offsets (scan) one tile ahead, so the value copy leaves as soon as its stage is free
         const int r = 2 * lane;
         auto rows = [&](int it) { return (int)min((int64_t)R, row_hi - (row_lo + (int64_t)(first + it * stride) * R)); };
         int64_t rb0 = 0, b0 = 0;      // raw reads of the tile after next; first node block of the next tile
         int rid0 = 0, rid1 = 0;
         uint32_t w0 = 0u, w1 = 0u, vb = 0u;  // the next tile's words and value bytes
         auto load = [&](int it) {
            const int64_t n0 = row_lo + (int64_t)(first + it * stride) * R;
            const int nloc = rows(it);
            rb0 = (COLS == kCompact ? ca.cbrp : brp)[n0];
            rid0 = r < nloc ? dict.sig[n0 + r] : 0, rid1 = r + 1 < nloc ? dict.sig[n0 + r + 1] : 0;
         };
         auto scan = [&](int it) {
            const int nloc = rows(it);
            constexpr int kd = kStencilD + (COLS == kCompact ? 1 : 0);  // the degree of the rows in the stage
            const int d0 = r < nloc ? sdict[rid0 * DS + kd] : 0;
            const int d1 = r + 1 < nloc ? sdict[rid1 * DS + kd] : 0;
            int incl = d0 + d1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
               const int v = __shfl_up_sync(0xffffffffu, incl, o);
               if (lane >= o) incl += v;
            }
            const uint32_t e0 = (uint32_t)(incl - d0 - d1);
            w0 = e0 | ((uint32_t)rid0 << 16), w1 = (e0 + d0) | ((uint32_t)rid1 << 16);
            vb = 32u * (uint32_t)__shfl_sync(0xffffffffu, incl, 31);  // the tile's blocks = brp[n0 + nloc] - brp[n0]
            b0 = rb0;
         };
         if (nmine > 0) load(0), scan(0);
         if (nmine > 1) load(1);
         for (int it = 0; it < nmine; ++it)
         {
            const int s = it % kTmaStages;
            if (it >= kTmaStages) mbar_wait(&empty[s], ((it / kTmaStages) - 1) & 1);
            unsigned char *st = smem + (size_t)s * stage_bytes;
            if (lane == 0 && vb)
            {
               mbar_expect_tx_only(&full[s], vb);
               bulk_g2s(st, values + 4 * b0, vb, &full[s]);
            }
            reinterpret_cast<uint2 *>(st + cap.vbytes)[lane] = make_uint2(w0, w1);
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
            if (it + 1 < nmine) scan(it + 1);
            if (it + 2 < nmine) load(it + 2);
         }
      }
      else if (lane == 0)
         for (int it = 0; it < nmine; ++it)
         {
            const int s = it % kTmaStages;
            if (it >= kTmaStages) mbar_wait(&empty[s], ((it / kTmaStages) - 1) & 1);
            const int64_t n0 = row_lo + (int64_t)(first + it * stride) * R;
            const int nloc = (int)min((int64_t)R, row_hi - n0);
            const int64_t b0 = brp[n0], b1 = brp[n0 + nloc];
            const uint32_t vb = (uint32_t)(32 * (b1 - b0));
            unsigned char *st = smem + (size_t)s * stage_bytes;
            {
               constexpr int CW = COLS == kC16 ? 2 : 4;                            // bytes per column index
               const int64_t c0 = b0 & ~(int64_t)(16 / CW - 1), p0 = n0 & ~(int64_t)1;
               const uint32_t cb = (uint32_t)((CW * (b1 - c0) + 15) & ~(int64_t)15);
               const uint32_t pb = (uint32_t)((8 * (n0 + nloc + 1 - p0) + 15) & ~(int64_t)15);
               mbar_expect_tx(&full[s], vb + cb + pb);
               if (vb) bulk_g2s(st, values + 4 * b0, vb, &full[s]);
               if (cb) bulk_g2s(st + cap.vbytes, static_cast<const unsigned char *>(bcol_any) + CW * c0, cb, &full[s]);
               bulk_g2s(st + cap.vbytes + cap.cbytes, brp + p0, pb, &full[s]);
            }
         }
   }
   else
   {  // ---- consumer warps: L lanes per node row pair ----
      constexpr int kSpmvLanes = L;
      const int sub = lane & (kSpmvLanes - 1);
      const double2 *x2 = reinterpret_cast<const double2 *>(x);
      for (int it = 0; it < nmine; ++it)
      {
         const int s = it % kTmaStages;
         const int64_t n0 = row_lo + (int64_t)(first + it * stride) * R;
         const int nloc = (int)min((int64_t)R, row_hi - n0);
         const unsigned char *st = smem + (size_t)s * stage_bytes;
         const double2 *sval = reinterpret_cast<const double2 *>(st);
         using col_t = typename std::conditional<COLS == kC32, int32_t, int16_t>::type;
         mbar_wait(&full[s], (it / kTmaStages) & 1);
         const col_t *scol = nullptr;
         const int64_t *sbrp = nullptr;
         int coff = 0;
         int64_t b0 = 0;
         if constexpr (!DICT)
         {
            scol = reinterpret_cast<const col_t *>(st + cap.vbytes);
            sbrp = reinterpret_cast<const int64_t *>(st + cap.vbytes + cap.cbytes) + (n0 & 1);
            b0 = sbrp[0];
            coff = (int)(b0 & (COLS == kC16 ? 7 : 3));
         }
#pragma unroll
         for (int pass = 0; pass < R * kSpmvLanes / kTmaConsumers; ++pass)
         {
            const int i = pass * (kTmaConsumers / kSpmvLanes) + tid / kSpmvLanes;
            int pb, deg, rdeg;  // rdeg: blocks of the row in the stage
            const col_t *cols;
            if constexpr (DICT)
            {
               const uint32_t w = i < nloc ? reinterpret_cast<const uint32_t *>(st + cap.vbytes)[i] : 0u;  // offset | id << 16
               pb = (int)(w & 0xffffu);
               cols = sdict + (w >> 16) * DS;
               deg = cols[kStencilD];
               rdeg = COLS == kCompact ? cols[kStencilD + 1] : deg;
            }
            else
            {
               pb = i < nloc ? (int)(sbrp[i] - b0) : 0;
               deg = i < nloc ? (int)(sbrp[i + 1] - b0) - pb : 0;
               cols = scol + coff + pb;
               rdeg = deg;
            }
            double y0 = 0., y1 = 0.;
            if (i < nloc)
            {
               const double2 *row0 = sval + 2 * pb, *row1 = row0 + rdeg;
               const double2 *xr = COLS != kC32 ? x2 + (n0 + i) : x2;  // 16-bit offsets and stencils are relative to the row's node
               // compact modes: position of slot t in the compact row (-1: dropped)
               const int16_t *cpos = COLS >= kCompactWrite ? reinterpret_cast<const int16_t *>(cols) + kStencilD + 2 : nullptr;
               double2 *cv0 = nullptr, *cv1 = nullptr;
               if constexpr (COLS == kCompactWrite)
               {
                  cv0 = reinterpret_cast<double2 *>(ca.cvalues) + 2 * ca.cbrp[n0 + i];
                  cv1 = cv0 + cols[kStencilD + 1];
               }
               int t = sub;
               for (; t + 2 * kSpmvLanes < deg; t += 3 * kSpmvLanes)
               {
                  const double2 v0 = x_block<COLS>(cpos, xr, cols, t), v1 = x_block<COLS>(cpos, xr, cols, t + kSpmvLanes),
                                v2 = x_block<COLS>(cpos, xr, cols, t + 2 * kSpmvLanes);
                  const double2 a0 = stage_block<COLS>(cpos, row0, t), a1 = stage_block<COLS>(cpos, row0, t + kSpmvLanes), a2 = stage_block<COLS>(cpos, row0, t + 2 * kSpmvLanes);
                  const double2 c0 = stage_block<COLS>(cpos, row1, t), c1 = stage_block<COLS>(cpos, row1, t + kSpmvLanes), c2 = stage_block<COLS>(cpos, row1, t + 2 * kSpmvLanes);
                  put<COLS>(cpos, cv0, cv1, ca.cbad, t, a0, c0), put<COLS>(cpos, cv0, cv1, ca.cbad, t + kSpmvLanes, a1, c1), put<COLS>(cpos, cv0, cv1, ca.cbad, t + 2 * kSpmvLanes, a2, c2);
                  y0 = __dadd_rn(y0, chain(a0, v0, a1, v1, a2, v2));
                  y1 = __dadd_rn(y1, chain(c0, v0, c1, v1, c2, v2));
               }
               if (t + kSpmvLanes < deg)
               {
                  const double2 v0 = x_block<COLS>(cpos, xr, cols, t), v1 = x_block<COLS>(cpos, xr, cols, t + kSpmvLanes);
                  const double2 a0 = stage_block<COLS>(cpos, row0, t), a1 = stage_block<COLS>(cpos, row0, t + kSpmvLanes);
                  const double2 c0 = stage_block<COLS>(cpos, row1, t), c1 = stage_block<COLS>(cpos, row1, t + kSpmvLanes);
                  put<COLS>(cpos, cv0, cv1, ca.cbad, t, a0, c0), put<COLS>(cpos, cv0, cv1, ca.cbad, t + kSpmvLanes, a1, c1);
                  y0 = __dadd_rn(y0, chain(a0, v0, a1, v1));
                  y1 = __dadd_rn(y1, chain(c0, v0, c1, v1));
               }
               else if (t < deg)
               {
                  const double2 v0 = x_block<COLS>(cpos, xr, cols, t);
                  const double2 a0 = stage_block<COLS>(cpos, row0, t), c0 = stage_block<COLS>(cpos, row1, t);
                  put<COLS>(cpos, cv0, cv1, ca.cbad, t, a0, c0);
                  y0 = __dadd_rn(y0, chain(a0, v0));
                  y1 = __dadd_rn(y1, chain(c0, v0));
               }
            }
#pragma unroll
            for (int o = kSpmvLanes / 2; o > 0; o >>= 1)
            {
               y0 += __shfl_xor_sync(0xffffffffu, y0, o);
               y1 += __shfl_xor_sync(0xffffffffu, y1, o);
            }
            if (i < nloc && sub == 0)
            {
               reinterpret_cast<double2 *>(y)[n0 + i] = make_double2(y0, y1);
               if (DOT)
               {
                  const double2 xi = x2[n0 + i];
                  part = __dadd_rn(part, __fma_rn(xi.x, y0, __dmul_rn(xi.y, y1)));
               }
            }
         }
         __syncwarp();
         if (lane == 0) mbar_arrive(&empty[s]);
      }
   }
   if (DOT) block_reduce_finish<kTmaThreads>(part, red, out, accumulate);
}

__global__ void diag_kernel(int64_t nnodes, const int64_t *__restrict__ brp, const uint8_t *__restrict__ dslot,
                            const double *__restrict__ values, double *__restrict__ diag)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   const int64_t bi = brp[I];
   const int deg = (int)(brp[I + 1] - bi), s = dslot[I];
   double2 d = make_double2(0., 0.);
   if (s < deg) d = make_double2(values[4 * bi + 2 * s], values[4 * bi + 2 * deg + 2 * s + 1]);
   reinterpret_cast<double2 *>(diag)[I] = d;
}

constexpr int kSpmvStages = 2;         // stages of the CSR modes: with the 16-bit layout they size every mode's grid
constexpr int kCompactStages = 3;      // kCompact: its smaller stages leave room for a third

struct SpmvShape
{
   SpmvTile cap;
   size_t smem;
   unsigned grid;
   int per_sm;
};

// Stage capacities, shared memory and grid of a mode over rr (grid 0: the tiles do not fit shared memory).  The stages
// of the index layout (the 16-bit one for the dictionary modes) size the grid: every mode but the 32-bit one runs the
// same CTAs over the same tiles, so that the per-CTA dot partials agree bit for bit.
static SpmvShape spmv_shape(const femb200_plan *p, const RowRange &rr, int R, int S, int COLS)
{
   SpmvShape sh{};
   const int ntiles = (int)cdiv(rr.hi - rr.lo, R);
   const int maxb = rr.tile_max[R == 32 ? 0 : 1];
   SpmvTile &cap = sh.cap;
   cap.vbytes = 32 * maxb;
   cap.cbytes = COLS != kC32 ? ((2 * (maxb + 8) + 15) & ~15) : ((4 * (maxb + 4) + 15) & ~15);
   cap.pbytes = ((8 * (R + 3) + 15) & ~15);
   sh.smem = (size_t)kSpmvStages * (cap.vbytes + cap.cbytes + cap.pbytes);
   const size_t budget = devinfo().smem_optin ? devinfo().smem_optin : 227 * 1024;
   if (sh.smem > budget) return sh;
   auto per_sm = [&](size_t smem) { return (int)std::max<size_t>(1, std::min<size_t>(7, (budget + 1024) / (smem + 1024))); };
   sh.per_sm = per_sm(sh.smem);
   sh.grid = (unsigned)std::min<int64_t>(ntiles, (int64_t)devinfo().sm_count * sh.per_sm);
   if (COLS >= kStencil)
   {  // S stages of values + one word per row (value offset | id << 16), then the dictionary
      if (COLS == kCompact) cap.vbytes = 32 * rr.ctile_max;
      cap.cbytes = 4 * R;
      cap.pbytes = 0;
      const int dbytes = COLS == kStencil ? 2 * kDictStride * p->nstencils : 2 * kCDictStride * p->ncompact;
      sh.smem = (size_t)S * (cap.vbytes + cap.cbytes) + ((dbytes + 15) & ~15);
      if (COLS >= kCompactWrite && (sh.smem > budget || per_sm(sh.smem) < sh.per_sm)) sh.grid = 0;  // fewer resident CTAs than the grid
   }
   return sh;
}

template <bool DOT, int R, int S, int L, int COLS>
static int spmv_tma_launch(const femb200_plan *p, const RowRange &rr, const double *d_values, const double *d_x,
                           double *d_y, const double *d_flag, double *d_dot_out, bool accumulate, cudaStream_t st,
                           SpmvCompactArgs ca = SpmvCompactArgs{nullptr, nullptr, nullptr})
{
   static_assert(R == 32 || R == 64, "RowRange::tile_max is measured for 32- and 64-row tiles");
   static_assert(R * L % kTmaConsumers == 0, "a tile must be a whole number of consumer passes");
   const int ntiles = (int)cdiv(rr.hi - rr.lo, R);
   const SpmvShape sh = spmv_shape(p, rr, R, S, COLS);
   if (!sh.grid) return -1;  // caller falls back to the direct kernel
   SpmvStencils dict{nullptr, nullptr, nullptr, 0};
   if (COLS == kStencil) dict = SpmvStencils{p->sig, p->stencil_off, p->stencil_deg, p->nstencils};
   if (COLS >= kCompactWrite) dict = SpmvStencils{p->csig, p->cdict, nullptr, p->ncompact};
   if (int rc = ensure_dynamic_smem<spmv_tma_kernel<DOT, R, S, L, COLS>>(sh.smem)) return rc;
   ReduceScratch red{nullptr, nullptr};
   if (DOT)
      if (int rc = reduce_scratch(sh.grid, st, &red)) return rc;
   spmv_tma_kernel<DOT, R, S, L, COLS><<<sh.grid, kTmaThreads, sh.smem, st>>>(
       rr.lo, rr.hi, p->brp, COLS == kC16 ? static_cast<const void *>(p->bcol16) : static_cast<const void *>(p->bcol), dict,
       d_values, d_x, d_y, d_flag, red, d_dot_out, sh.cap, ntiles, accumulate, ca);
   FEMB_LAUNCH_CHECK();
   return 0;
}

template <int COLS>
static int spmv_tma_dispatch(const femb200_plan *p, const RowRange &rr, const double *d_values, const double *d_x,
                             double *d_y, const double *d_flag, double *d_dot_out, bool accumulate, cudaStream_t st,
                             SpmvCompactArgs ca = SpmvCompactArgs{nullptr, nullptr, nullptr})
{
   return d_dot_out
              ? spmv_tma_launch<true, 64, kSpmvStages, 4, COLS>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st, ca)
              : spmv_tma_launch<false, 64, kSpmvStages, 4, COLS>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st, ca);
}

bool spmv_compact_ready(femb200_plan *p, const RowRange &rr)
{
   if (!p->csig || p->opt_spmv_compact != 0 || p->opt_spmv_path != 0 || !p->sig || p->opt_spmv_cols != 0 ||
       rr.hi <= rr.lo || rr.ctile_max <= 0 || p->cvalues_failed)
      return false;
   if (!spmv_shape(p, rr, 64, kSpmvStages, kCompactWrite).grid || !spmv_shape(p, rr, 64, kCompactStages, kCompact).grid)
      return false;
   if (p->cvalues) return true;
   std::lock_guard<std::mutex> lock(p->range_mtx);
   if (p->cvalues) return true;
   if (cudaMalloc(&p->cbad, sizeof(int)) != cudaSuccess || cudaMalloc(&p->cvalues, 32 * (size_t)p->nkept) != cudaSuccess)
   {  // not enough device memory: this plan's solves keep streaming the CSR values
      cudaGetLastError();
      cudaFree(p->cbad), cudaFree(p->cvalues);
      p->cbad = nullptr, p->cvalues = nullptr;
      p->cvalues_failed = true;
      return false;
   }
   p->bytes += 32 * (size_t)p->nkept + sizeof(int);
   return true;
}

// y = A x on the node rows of rr (+ d_dot_out (+)= <x, y> over those rows; no-op when *d_flag != 0).
// Default: 64-row tiles, 2 stages (3 CTAs per SM), 4 lanes per row: 0.59 ms on the n = 1448 P2 matrix against
// 0.99 ms with 3 stages and 8 lanes (profiles/r1_summary.md).  Columns: stencil ids when the plan has them, else
// 16-bit offsets, else 32-bit indices (option spmv_cols forces the latter two).  Tiles too large for shared memory,
// and plans with spmv_path = 1, take the direct kernel.
int spmv_launch(const femb200_plan *p, const RowRange &rr, const double *d_values, const double *d_x, double *d_y,
                const double *d_flag, double *d_dot_out, bool accumulate, cudaStream_t st, int compact)
{
   const int64_t nrows = rr.hi - rr.lo;
   if (nrows <= 0)
   {
      if (d_dot_out && !accumulate) FEMB_CUDA(cudaMemsetAsync(d_dot_out, 0, sizeof(double), st));
      return 0;
   }
   if (compact)
   {  // spmv_compact_ready() has checked the plan, the stages and the buffers; the fused dot is always requested
      FEMB_CHECK(d_dot_out && p->cvalues, "spmv: the compact modes need the fused dot and a compact copy");
      SpmvCompactArgs ca{p->cbrp, p->cvalues, p->cbad};
      if (compact == 1)
         return spmv_tma_launch<true, 64, kSpmvStages, 4, kCompactWrite>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out,
                                                                          accumulate, st, ca);
      if (int rc = spmv_tma_launch<true, 64, kCompactStages, 4, kCompact>(p, rr, p->cvalues, d_x, d_y, d_flag, d_dot_out,
                                                                          accumulate, st, ca))
         return rc;
      // the CSR values when the first apply found a dropped block that is not zero (a no-op otherwise)
      return spmv_tma_dispatch<kStencil>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st, ca);
   }
   if (p->opt_spmv_path == 0)
   {
      int rc;
      if (p->sig && p->opt_spmv_cols == 0)
         rc = spmv_tma_dispatch<kStencil>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st);
      else if (p->bcol16 && p->opt_spmv_cols != 1)
         rc = spmv_tma_dispatch<kC16>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st);
      else
         rc = spmv_tma_dispatch<kC32>(p, rr, d_values, d_x, d_y, d_flag, d_dot_out, accumulate, st);
      if (rc >= 0) return rc;
   }
   const unsigned grid = (unsigned)cdiv(nrows * kSpmvLanes, kSpmvThreads);
   if (d_dot_out)
   {
      ReduceScratch red;
      if (int rc = reduce_scratch(grid, st, &red)) return rc;
      spmv_kernel<true><<<grid, kSpmvThreads, 0, st>>>(rr.lo, rr.hi, p->brp, p->bcol, d_values, d_x, d_y, d_flag, red,
                                                        d_dot_out, accumulate);
   }
   else
      spmv_kernel<false><<<grid, kSpmvThreads, 0, st>>>(rr.lo, rr.hi, p->brp, p->bcol, d_values, d_x, d_y, d_flag,
                                                         ReduceScratch{nullptr, nullptr}, nullptr);
   FEMB_LAUNCH_CHECK();
   return 0;
}

}  // namespace femb

using namespace femb;

extern "C" int femb200_spmv(const femb200_plan *p, const double *d_values, const double *d_x, double *d_y, void *stream)
{
   FEMB_CHECK(p && d_values && d_x && d_y, "spmv: null argument");
   FEMB_CHECK(d_x != d_y, "spmv: x and y must not alias");
   RowRange rr;
   if (int rc = plan_row_range(p, 0, p->nnodes, &rr)) return rc;
   return spmv_launch(p, rr, d_values, d_x, d_y, nullptr, nullptr, false, as_stream(stream));
}

extern "C" int femb200_spmv_dot(const femb200_plan *p, const double *d_values, const double *d_x, double *d_y,
                                double *d_dot, void *stream)
{
   FEMB_CHECK(p && d_values && d_x && d_y && d_dot, "spmv_dot: null argument");
   FEMB_CHECK(d_x != d_y, "spmv_dot: x and y must not alias");
   RowRange rr;
   if (int rc = plan_row_range(p, 0, p->nnodes, &rr)) return rc;
   return spmv_launch(p, rr, d_values, d_x, d_y, nullptr, d_dot, false, as_stream(stream));
}

// y = A x on the node rows [row_lo, row_hi) (the rows a rank owns, or the rows next to its ghosts); rows
// outside are left untouched.  d_dot (or NULL) receives <x, y> over those rows, added to its content when
// `accumulate`; d_flag (or NULL): no-op when *d_flag != 0 (converged CG).  The first call with a range that
// does not start on a 64-row boundary measures its tiling (synchronises the device once).
extern "C" int femb200_spmv_rows(const femb200_plan *p, const double *d_values, const double *d_x, double *d_y,
                                 int64_t row_lo, int64_t row_hi, double *d_dot, int accumulate, const double *d_flag,
                                 void *stream)
{
   FEMB_CHECK(p && d_values && d_x && d_y, "spmv_rows: null argument");
   FEMB_CHECK(d_x != d_y, "spmv_rows: x and y must not alias");
   RowRange rr;
   if (int rc = plan_row_range(p, row_lo, row_hi, &rr)) return rc;
   return spmv_launch(p, rr, d_values, d_x, d_y, d_flag, d_dot, accumulate != 0, as_stream(stream));
}

extern "C" int femb200_extract_diagonal(const femb200_plan *p, const double *d_values, double *d_diag, void *stream)
{
   FEMB_CHECK(p && d_values && d_diag, "extract_diagonal: null argument");
   const int T = 256;
   diag_kernel<<<(unsigned)cdiv(p->nnodes, T), T, 0, as_stream(stream)>>>(p->nnodes, p->brp, p->dslot, d_values, d_diag);
   FEMB_LAUNCH_CHECK();
   return 0;
}
