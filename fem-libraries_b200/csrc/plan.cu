// plan.cu -- sparsity pattern and gather maps, built on the device from the
// cell->dof map alone.
//
// Role in the reference: dolfinx::fem::petsc::create_matrix(*J_form) (F.cc:688),
// which builds the CSR structure once before the Newton loop.  The pattern is the
// dolfinx convention (SURVEY.md 8c): rows in dof order, columns ascending and
// unique, structural, bs = 2.  Because every scalar row 2I+i of node I has the
// same column set {2J, 2J+1 : J in adj(I)}, the pattern is stored once per node
// ("block CSR": brp/bcol) and the scalar CSR is a closed-form expansion:
//     rowptr[2I]   = 4 brp[I]
//     rowptr[2I+1] = 4 brp[I] + 2 deg(I)
//     colidx[rowptr[2I+i] + 2s + k] = 2 bcol[brp[I]+s] + k
#include "plan.cuh"

namespace femb {

constexpr int kMaxDeg = 96;  // block degree cap of the builder (thread-local scratch)

// --- input validation: every dof / geometry index inside [0, nnodes) ----------------------------
__global__ void k_check_range(int64_t n, const int32_t *__restrict__ idx, int32_t nnodes, int32_t *__restrict__ bad)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n && (idx[i] < 0 || idx[i] >= nnodes)) atomicOr(bad, 1);
}

// --- node -> cell visit lists -------------------------------------------------
__global__ void k_count_visits(int64_t nvis, const int32_t *__restrict__ dofmap, int32_t *__restrict__ cnt)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < nvis) atomicAdd(&cnt[dofmap[i]], 1);
}

__global__ void k_fill_visits(int64_t nvis, int nd, const int32_t *__restrict__ dofmap,
                              const int32_t *__restrict__ nptr, int32_t *__restrict__ cursor,
                              uint32_t *__restrict__ tmp)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= nvis) return;
   const int32_t I = dofmap[i];
   const int32_t p = atomicAdd(&cursor[I], 1);
   const uint32_t e = (uint32_t)(i / nd), a = (uint32_t)(i % nd);
   tmp[nptr[I] + p] = (e << 4) | a;
}

// atomics fill each list in arbitrary order: sort (ascending cell id) for determinism
__global__ void k_sort_visits(int64_t nnodes, const int32_t *__restrict__ nptr, uint32_t *__restrict__ tmp)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   const int32_t lo = nptr[I], hi = nptr[I + 1];
   for (int32_t i = lo + 1; i < hi; ++i)
   {
      const uint32_t v = tmp[i];
      int32_t j = i - 1;
      while (j >= lo && tmp[j] > v)
      {
         tmp[j + 1] = tmp[j];
         --j;
      }
      tmp[j + 1] = v;
   }
}

// Triangles: re-order the visits of every VERTEX row rotationally (a fan around the node): cell k
// shares one of its two fan edges (I, V) with cell k+1, so the contribution of consecutive visits to
// that edge's columns can be carried in registers by the assembly kernel instead of being read back
// from the staging image (see k_fast_records).  Orientation-agnostic: the walk leaves every cell by
// the fan vertex it did not enter by.  It starts at a boundary cell of an open fan (a fan vertex
// that belongs to one cell only; the smallest such vertex), else at the smallest fan vertex (closed
// fan; the lower of its two cells); where the walk breaks it restarts at the smallest remaining
// cell.  Edge rows (two cells) keep ascending cell order.  The order depends on the relative order
// of node / cell numbers only: deterministic, and identical on every partition of a mesh.
__global__ void k_order_visits(int64_t nnodes, int nd, const int32_t *__restrict__ dofmap,
                               const int32_t *__restrict__ nptr, uint32_t *__restrict__ tmp)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   const int32_t lo = nptr[I];
   const int cnt = nptr[I + 1] - lo;
   if (cnt < 2 || cnt > kAsmLevels) return;
   uint32_t v[kAsmLevels];
   int32_t p1[kAsmLevels], p2[kAsmLevels];
   for (int k = 0; k < cnt; ++k)
   {
      v[k] = tmp[lo + k];
      const int a = (int)(v[k] & 15u);
      if (a >= 3) return;  // an edge row
      const int64_t e = v[k] >> 4;
      p1[k] = dofmap[e * nd + (a + 1) % 3];
      p2[k] = dofmap[e * nd + (a + 2) % 3];
   }
   auto occurrences = [&](int32_t vert) {
      int n = 0;
      for (int j = 0; j < cnt; ++j) n += (p1[j] == vert) + (p2[j] == vert);
      return n;
   };
   // start cell and entry vertex
   int cur = -1;
   int32_t entry = 0;
   for (int pass = 0; pass < 2 && cur < 0; ++pass)  // pass 0: open-fan ends, pass 1: any vertex
      for (int k = 0; k < cnt; ++k)
         for (int side = 0; side < 2; ++side)
         {
            const int32_t vert = side ? p2[k] : p1[k];
            if (pass == 0 && occurrences(vert) != 1) continue;
            if (cur < 0 || vert < entry) cur = k, entry = vert;
         }
   uint32_t used = 0u;
   for (int out = 0; out < cnt; ++out)
   {
      tmp[lo + out] = v[cur];
      used |= 1u << cur;
      const int32_t exitv = (entry == p1[cur]) ? p2[cur] : p1[cur];
      int nxt = -1;
      for (int j = 0; j < cnt; ++j)
         if (!((used >> j) & 1u) && nxt < 0 && (p1[j] == exitv || p2[j] == exitv)) nxt = j;
      entry = exitv;
      if (nxt < 0)  // the walk breaks: smallest remaining cell (v[] is in ascending cell order)
         for (int j = 0; j < cnt; ++j)
            if (!((used >> j) & 1u) && nxt < 0) nxt = j, entry = p1[j];
      cur = nxt;
   }
}

// --- neighbour sets -------------------------------------------------------------
// sorted unique neighbour nodes of row node I into loc[]; returns the count, or
// -1 when kMaxDeg is exceeded
__device__ inline int gather_neighbours(int64_t I, int nd, const int32_t *__restrict__ dofmap,
                                        const int32_t *__restrict__ nptr, const uint32_t *__restrict__ vis,
                                        int32_t *loc)
{
   int deg = 0;
   for (int32_t k = nptr[I]; k < nptr[I + 1]; ++k)
   {
      const int64_t e = vis[k] >> 4;
      for (int b = 0; b < nd; ++b)
      {
         const int32_t J = dofmap[e * nd + b];
         // sorted insert with de-duplication
         int lo = 0, hi = deg;
         while (lo < hi)
         {
            const int mid = (lo + hi) >> 1;
            if (loc[mid] < J)
               lo = mid + 1;
            else
               hi = mid;
         }
         if (lo < deg && loc[lo] == J) continue;
         if (deg == kMaxDeg) return -1;
         for (int t = deg; t > lo; --t) loc[t] = loc[t - 1];
         loc[lo] = J;
         ++deg;
      }
   }
   return deg;
}

__global__ void k_degree(int64_t nnodes, int nd, const int32_t *__restrict__ dofmap, const int32_t *__restrict__ nptr,
                         const uint32_t *__restrict__ vis, int32_t *__restrict__ deg, int32_t *__restrict__ flags)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   int32_t loc[kMaxDeg];
   const int d = gather_neighbours(I, nd, dofmap, nptr, vis, loc);
   if (d < 0)
   {
      atomicOr(flags, 1);
      deg[I] = 0;
   }
   else
   {
      deg[I] = d;
      atomicMax(flags + 1, d);
   }
}

__global__ void k_fill_cols(int64_t nnodes, int nd, const int32_t *__restrict__ dofmap,
                            const int32_t *__restrict__ nptr, const uint32_t *__restrict__ vis,
                            const int64_t *__restrict__ brp, int32_t *__restrict__ bcol, uint8_t *__restrict__ dslot)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   int32_t loc[kMaxDeg];
   const int d = gather_neighbours(I, nd, dofmap, nptr, vis, loc);
   const int64_t base = brp[I];
   int ds = 255;
   for (int s = 0; s < d; ++s)
   {
      bcol[base + s] = loc[s];
      if (loc[s] == I) ds = s;
   }
   dslot[I] = (uint8_t)ds;
}

// local dof of ROTATED column t for a row with local index a: the row's own vertex / edge becomes
// number 0 of its group (vertices m, m+1, m+2 then edges 3+m, 3+m+1, 3+m+2, indices mod 3)
__device__ __forceinline__ int rotated_local(int t, int a)
{
   const int m = (a >= 3) ? a - 3 : a;
   const int tt = (t >= 3) ? t - 3 : t;
   int b = m + tt;
   b = (b >= 3) ? b - 3 : b;
   return (t >= 3) ? b + 3 : b;
}

// --- slot map: position of every local dof b of visit (I, e, a) in block row I ---
__global__ void k_fill_slots(int64_t nnodes, int nd, bool rotated, const int32_t *__restrict__ dofmap,
                             const int32_t *__restrict__ nptr, const uint32_t *__restrict__ vis,
                             const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                             VisitRec *__restrict__ vrec)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   const int64_t base = brp[I];
   const int deg = (int)(brp[I + 1] - base);
   uint32_t touched[(kMaxDeg + 31) / 32];
   for (int t = 0; t < (kMaxDeg + 31) / 32; ++t) touched[t] = 0u;
   for (int32_t k = nptr[I]; k < nptr[I + 1]; ++k)
   {
      VisitRec r;
      r.e = vis[k] >> 4;
      r.a = (uint8_t)(vis[k] & 15u);
      r.first = 0;
      r.slot8 = 0;
      for (int b = 0; b < 8; ++b) r.slot[b] = 0;
      for (int t = 0; t < nd; ++t)
      {  // stored position t: triangles keep the columns in ROTATED order (plan.cuh), quads in natural order
         const int b = rotated ? rotated_local(t, (int)r.a) : t;
         const int32_t J = dofmap[(int64_t)r.e * nd + b];
         int lo = 0, hi = deg;
         while (lo < hi)
         {
            const int mid = (lo + hi) >> 1;
            if (bcol[base + mid] < J)
               lo = mid + 1;
            else
               hi = mid;
         }
         if (t < 8)
            r.slot[t] = (uint8_t)lo;
         else
            r.slot8 = (uint8_t)lo;
         if (!((touched[lo >> 5] >> (lo & 31)) & 1u))
         {
            touched[lo >> 5] |= 1u << (lo & 31);
            r.first |= (uint16_t)(1u << t);
         }
      }
      vrec[k] = r;
   }
}

// --- tile-sorted storage order of the visit records -------------------------------------
// one CTA of kAsmR threads per tile: rank the nodes by decreasing visit count (ties by index),
// write perm and the level offsets, move every record to nptr[n0] + voff[j] + rank
__global__ void __launch_bounds__(kAsmR)
k_tile_sort(int64_t nnodes, const int32_t *__restrict__ nptr, const VisitRec *__restrict__ src,
            VisitRec *__restrict__ dst, uint8_t *__restrict__ perm, uint16_t *__restrict__ voff,
            int32_t *__restrict__ flags)
{
   __shared__ int s_cnt[kAsmR], s_off[kAsmLevels + 1];
   const int i = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR, node = n0 + i;
   const int32_t k0 = node < nnodes ? nptr[node] : 0;
   const int cnt = node < nnodes ? nptr[node + 1] - k0 : -1;
   s_cnt[i] = cnt;
   __syncthreads();
   int rank = 0;
   for (int t = 0; t < kAsmR; ++t) rank += (s_cnt[t] > cnt) || (s_cnt[t] == cnt && t < i);
   perm[n0 + rank] = (uint8_t)i;  // padding nodes of the last tile rank last (cnt = -1)
   if (cnt > kAsmLevels) atomicOr(flags, 1);
   if (i <= kAsmLevels)
   {  // s_off[j] = records in levels < j = sum over nodes of min(cnt, j)
      int o = 0;
      for (int t = 0; t < kAsmR; ++t) o += max(0, min(s_cnt[t], i));
      s_off[i] = o;
   }
   __syncthreads();
   if (i < kAsmLevels) voff[(int64_t)blockIdx.x * kAsmLevels + i] = (uint16_t)s_off[i];
   const int32_t vbase = nptr[n0];
   for (int j = 0; j < cnt && j < kAsmLevels; ++j) dst[vbase + s_off[j] + rank] = src[k0 + j];
}

// --- fast-path records (plan.cuh): staging addresses resolved at plan time ----------------
// one CTA of kAsmR threads per tile, thread = rank.  Put semantics of the fast kernel:
//  * the diagonal block (position 0 of a vertex row, 3 of an edge row) is accumulated in registers
//    over all visits and stored once after the last one: never "put";
//  * every visit has two "sides", the columns that go with its two other vertices 1' and 2':
//    side 0 = positions (1, 5), side 1 = positions (2, 4) for a vertex row (vertex, midpoint of the
//    fan edge); positions 1 and 2 (the two ends) for an edge row.  The kernel ALWAYS adds its carry
//    registers to side 0 and, when the carry-out bit is set, keeps side 1 (vertex row) / both ends
//    (edge row) in registers for the next visit instead of putting them.  To make that static
//    pairing hold, this pass may FLIP a visit: vertices 1' and 2' (hence positions 1 <-> 2, 4 <-> 5)
//    exchange their roles, which the closed form of the element matrix allows (it is symmetric
//    under relabelling); the record carries the local vertex numbers of 1' and 2';
//  * first-touch bits describe the puts that actually happen, in visit order.
// The pairing is verified here on the slots; where it does not hold the columns are put as usual.
__global__ void __launch_bounds__(kAsmR)
k_fast_records(int64_t nnodes, int nd, const int32_t *__restrict__ nptr, const int64_t *__restrict__ brp,
               const uint8_t *__restrict__ perm, const uint16_t *__restrict__ voff, const VisitRec *__restrict__ vrec,
               int flevels, uint4 *__restrict__ frec, uint8_t *__restrict__ tcnt)
{
   const int rank = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR;
   const int nloc = (int)min((int64_t)kAsmR, nnodes - n0);
   if (rank >= nloc) return;
   const int64_t node = n0 + perm[n0 + rank];
   const int cnt = nptr[node + 1] - nptr[node];
   tcnt[n0 + rank] = (uint8_t)cnt;
   const int deg = (int)(brp[node + 1] - brp[node]);
   // first 16-byte unit of scalar row 0 in the tile image: the image starts at the tile's offset inside its 128-byte line
   const int r0 = (int)((2 * brp[n0]) & 7) + 2 * (int)(brp[node] - brp[n0]);
   const int32_t vbase = nptr[n0];
   const uint16_t *vo = voff + (int64_t)blockIdx.x * kAsmLevels;
   uint32_t touched[(kMaxDeg + 31) / 32];
   for (int t = 0; t < (kMaxDeg + 31) / 32; ++t) touched[t] = 0u;
   const bool p2 = nd > 3;
   bool cin = false;
   int carry_v = -1, carry_e = -1;  // slots of the columns held in the carry registers
   for (int j = 0; j < cnt; ++j)
   {
      const VisitRec r = vrec[(int64_t)vbase + vo[j] + rank];
      const bool vert = r.a < 3;
      const int diag = vert ? 0 : 3;
      const int m = vert ? r.a : r.a - 3;
      VisitRec q = r;
      const bool has_next = j + 1 < cnt;
      if (has_next) q = vrec[(int64_t)vbase + vo[j + 1] + rank];
      const bool same_kind = has_next && ((q.a < 3) == vert);
      // does side `rs` of this visit (natural numbering) coincide with a side of the next visit?
      auto side_matches_next = [&](int rs) {
         if (!same_kind) return false;
         for (int qs = 0; qs < 2; ++qs)
            if (r.slot[1 + rs] == q.slot[1 + qs] && (!p2 || !vert || r.slot[5 - rs] == q.slot[5 - qs])) return true;
         return false;
      };
      int flip = 0;
      bool cout = false;
      if (vert)
      {
         if (cin)
         {  // side 0 must be the side that is in the carry registers
            flip = (r.slot[1] == carry_v && (!p2 || r.slot[5] == carry_e)) ? 0 : 1;
            cout = side_matches_next(1 - flip);  // natural side 1 - flip becomes side 1
         }
         else if (side_matches_next(1))
            cout = true;
         else if (side_matches_next(0))
            cout = true, flip = 1;
      }
      else
      {
         if (cin) flip = (r.slot[1] == carry_v) ? 0 : 1;  // see the ends in the order of the first cell
         else
            cout = same_kind && ((r.slot[1] == q.slot[1] && r.slot[2] == q.slot[2]) ||
                                 (r.slot[1] == q.slot[2] && r.slot[2] == q.slot[1]));
      }
      // positions after the flip
      int sl[6];
      for (int t = 0; t < 6; ++t) sl[t] = r.slot[t];
      if (flip)
      {
         sl[1] = r.slot[2], sl[2] = r.slot[1];
         sl[4] = r.slot[5], sl[5] = r.slot[4];
      }
      const int i1 = (m + (flip ? 2 : 1)) % 3, i2 = (m + (flip ? 1 : 2)) % 3;  // local numbers of 1', 2'
      uint32_t first = 0u;
      int bit = 0;
      for (int t = 0; t < nd && t < 6; ++t)
      {
         if (t == diag) continue;
         const bool carried = cout && (vert ? (t == 2 || t == 4) : (t == 1 || t == 2));
         if (!carried && !((touched[sl[t] >> 5] >> (sl[t] & 31)) & 1u))
         {
            touched[sl[t] >> 5] |= 1u << (sl[t] & 31);
            first |= 1u << bit;
         }
         ++bit;
      }
      // one record per visit (plan.cuh): positions of row 0, the row-1 thread adds the block degree
      uint32_t pos[6] = {0u, 0u, 0u, 0u, 0u, 0u};
      for (int t = 0; t < nd && t < 6; ++t) pos[t] = (uint32_t)(r0 + sl[t]);
      frec[((int64_t)blockIdx.x * flevels + j) * kAsmR + rank] =
         make_uint4(r.e | ((uint32_t)cnt << 28),
                    pos[0] | (pos[1] << 11) | ((first & 0x1fu) << 22) | (cout ? 1u << 27 : 0u) | (vert ? 0u : 1u << 28) | ((uint32_t)i1 << 29),
                    pos[2] | (pos[3] << 11) | ((uint32_t)deg << 22) | ((uint32_t)i2 << 29), pos[4] | (pos[5] << 11));
      cin = cout;
      if (cout) carry_v = vert ? sl[2] : sl[1], carry_e = vert ? (p2 ? sl[4] : -1) : sl[2];
   }
}

// --- slot map of the damage-record stage of the fast kernel ----------------------------------
// one CTA of kAsmR threads per tile, thread = rank: the distinct cells of the tile's visits get slot numbers
// 0, 1, .. (shared hash table, first come first served: the numbering only decides where a record sits in the stage);
// the slot goes into the tile's fast records and, as (tile << 10 | slot), into the cell's reference list cref.  Cells
// beyond the capacity of the stage keep slot 0x3ff and are read from global memory by their visits.
__global__ void __launch_bounds__(kAsmR)
k_tile_cells(int64_t nnodes, int flevels, int cap, uint4 *__restrict__ frec, const uint8_t *__restrict__ tcnt,
             uint32_t *__restrict__ cref, int32_t *__restrict__ crefcnt)
{
   constexpr int H = 2048;  // >= 2 x the visits of a tile (kAsmR rows x 15 levels)
   __shared__ int32_t key[H], val[H];
   __shared__ int next;
   const int rank = threadIdx.x;
   const int64_t n0 = (int64_t)blockIdx.x * kAsmR;
   for (int t = rank; t < H; t += kAsmR) key[t] = -1;
   if (rank == 0) next = 0;
   __syncthreads();
   const int cnt = n0 + rank < nnodes ? (int)tcnt[n0 + rank] : 0;
   uint4 *rec = frec + ((int64_t)blockIdx.x * flevels) * kAsmR + rank;
   for (int j = 0; j < cnt; ++j)
   {
      const int32_t e = (int32_t)(rec[(int64_t)j * kAsmR].x & 0x0fffffffu);
      unsigned h = ((unsigned)e * 2654435761u) >> 21;  // 11 bits
      for (;;)
      {
         const int32_t prev = atomicCAS(&key[h], -1, e);
         if (prev == -1)
         {  // this thread inserted the cell: it hands out the slot
            const int s = atomicAdd(&next, 1);
            const int v = s < cap ? s : 0x3ff;
            if (cap > 0)
            {
               const int k = atomicAdd(&crefcnt[e], 1);  // a triangle has at most 6 nodes, hence at most 6 tiles
               if (k < 6) cref[8 * (int64_t)e + k] = ((uint32_t)blockIdx.x << 10) | (uint32_t)v;
            }
            val[h] = v;
            break;
         }
         if (prev == e) break;
         h = (h + 1) & (H - 1);
      }
   }
   __syncthreads();
   for (int j = 0; j < cnt; ++j)
   {
      uint4 r = rec[(int64_t)j * kAsmR];
      const int32_t e = (int32_t)(r.x & 0x0fffffffu);
      unsigned h = ((unsigned)e * 2654435761u) >> 21;
      while (key[h] != e) h = (h + 1) & (H - 1);
      r.w = (r.w & 0x003fffffu) | ((uint32_t)val[h] << 22);
      rec[(int64_t)j * kAsmR] = r;
   }
}

__global__ void k_tile_hdr(int64_t nnodes, int64_t ntiles, const int32_t *__restrict__ nptr,
                           const int64_t *__restrict__ brp, const uint16_t *__restrict__ voff, TileHdr *__restrict__ hdr,
                           int32_t *__restrict__ maxcnt)
{
   const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (t >= ntiles) return;
   const int64_t n0 = t * kAsmR, n1 = min(n0 + (int64_t)kAsmR, nnodes);
   TileHdr h;
   h.b0 = brp[n0];
   h.vbase = nptr[n0];
   h.nvis = nptr[n1] - nptr[n0];
   h.units = 2 * (int32_t)(brp[n1] - brp[n0]);
   h.pad = 0;
   for (int j = 0; j < kAsmLevels; ++j) h.voff[j] = voff[t * kAsmLevels + j];
   for (int j = 0; j < 4; ++j) h.pad2[j] = 0;
   hdr[t] = h;
   int m = 0;
   for (int64_t i = n0; i < n1; ++i) m = max(m, nptr[i + 1] - nptr[i]);
   atomicMax(maxcnt, m);
}

// --- largest staging tile (in node blocks) for each candidate tile height R ------
__global__ void k_tile_max(int64_t nnodes, const int64_t *__restrict__ brp, int32_t *__restrict__ out)
{
   const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
   for (int r = 0; r < kNumTileR; ++r)
   {
      const int64_t n0 = t * tile_r(r);
      if (n0 < nnodes)
      {
         const int64_t n1 = min(n0 + (int64_t)tile_r(r), nnodes);
         atomicMax(out + r, (int32_t)(brp[n1] - brp[n0]));
      }
   }
}

// largest tile of the tiling [lo + t R, lo + (t + 1) R) of the row range [lo, hi)
__global__ void k_range_tile_max(int64_t lo, int64_t hi, int R, const int64_t *__restrict__ brp, int32_t *__restrict__ out)
{
   const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   const int64_t n0 = lo + t * R;
   if (n0 < hi) atomicMax(out, (int32_t)(brp[min(n0 + (int64_t)R, hi)] - brp[n0]));
}

// --- scalar CSR expansion ---------------------------------------------------------
// 16-bit relative column indices of the block pattern for the SpMV (spmv.cu): bcol16[k] = bcol[k] - I for the blocks
// of node row I; *bad is set when an offset does not fit (the plan then keeps the 32-bit indices only)
__global__ void k_cols16(int64_t nnodes, const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                         int16_t *__restrict__ bcol16, int32_t *__restrict__ bad)
{
   const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;  // eight lanes per node row
   const int lane = threadIdx.x & 7;
   if (w >= nnodes) return;
   const int64_t b0 = brp[w], b1 = brp[w + 1];
   for (int64_t k = b0 + lane; k < b1; k += 8)
   {
      const int64_t d = (int64_t)bcol[k] - w;
      if (d < -32768 || d > 32767) *bad = 1;
      bcol16[k] = (int16_t)d;
   }
}

__global__ void k_scalar_csr(int64_t nnodes, const int64_t *__restrict__ brp, const int32_t *__restrict__ bcol,
                             int64_t *__restrict__ rowptr, int32_t *__restrict__ colidx)
{
   // one warp per node row pair: coalesced colidx writes
   const int64_t I = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
   const int lane = threadIdx.x & 31;
   if (I >= nnodes) return;
   const int64_t b0 = brp[I];
   const int deg = (int)(brp[I + 1] - b0);
   if (lane == 0)
   {
      rowptr[2 * I] = 4 * b0;
      rowptr[2 * I + 1] = 4 * b0 + 2 * deg;
      if (I == nnodes - 1) rowptr[2 * nnodes] = 4 * brp[nnodes];
   }
   for (int t = lane; t < 4 * deg; t += 32)
   {  // entry t of the 4*deg scalars of node I: row r = t / (2 deg), then (s, k)
      const int r = t / (2 * deg), w = t - r * 2 * deg;
      colidx[4 * b0 + t] = 2 * bcol[b0 + (w >> 1)] + (w & 1);
   }
}

// --- Dirichlet list ---------------------------------------------------------------
__global__ void k_bc_nodes(int64_t nnodes, const uint8_t *__restrict__ bc, int32_t *__restrict__ list,
                           int32_t *__restrict__ count)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes) return;
   if (bc[2 * I] | bc[2 * I + 1])
   {
      const int32_t p = atomicAdd(count, 1);
      if (list) list[p] = (int32_t)I;
   }
}

// mark[I] = 1 for every node I in the row of a constrained node J (symmetric pattern: the rows that have column J)
__global__ void k_mark_lift_rows(int nbc, const int32_t *__restrict__ bc_nodes, const int64_t *__restrict__ brp,
                                 const int32_t *__restrict__ bcol, uint8_t *__restrict__ mark)
{
   const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
   if (w >= nbc) return;
   const int64_t J = bc_nodes[w], b0 = brp[J], b1 = brp[J + 1];
   for (int64_t k = b0 + lane; k < b1; k += 32) mark[bcol[k]] = 1;
}
__global__ void k_compact_marked(int64_t nnodes, const uint8_t *__restrict__ mark, int32_t *__restrict__ list,
                                 int32_t *__restrict__ count)
{
   const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (I >= nnodes || !mark[I]) return;
   const int32_t p = atomicAdd(count, 1);
   if (list) list[p] = (int32_t)I;
}

template <typename T>
static int dev_alloc(T **p, size_t n, size_t *acc)
{
   *p = nullptr;
   const size_t bytes = sizeof(T) * (n ? n : 1);
   FEMB_CUDA(cudaMalloc(p, bytes));
   *acc += bytes;
   return 0;
}

}  // namespace femb

using namespace femb;

extern "C" void femb200_plan_destroy(femb200_plan *p)
{
   if (!p) return;
   cudaFree(p->nptr);
   cudaFree(p->vrec);
   cudaFree(p->frec);
   cudaFree(p->tcnt);
   cudaFree(p->thdr);
   cudaFree(p->perm);
   cudaFree(p->voff);
   cudaFree(p->brp);
   cudaFree(p->bcol);
   cudaFree(p->bcol16);
   cudaFree(p->dslot);
   cudaFree(p->bc);
   cudaFree(p->bc_nodes);
   cudaFree(p->lift_nodes);
   cudaFree(p->norm_partials);
   cudaFree(p->cellrec);
   cudaFree(p->cref);
   cudaFree(p->tdam);
   cudaFree(p->dmg_counter);
   if (p->dmg_count) cudaFreeHost(p->dmg_count);
   cudaFree(p->celld);
   cudaFree(p->celld_count);
   delete p;
}

extern "C" int femb200_plan_create(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap,
                                   const int32_t *d_xdofmap, void *stream, femb200_plan **out)
{
   FEMB_CHECK(out != nullptr, "plan_create: out is null");
   *out = nullptr;
   FEMB_CHECK(etype >= FEMB200_P1 && etype <= FEMB200_Q1, "plan_create: unknown element family %d", etype);
   FEMB_CHECK(nnodes > 0 && ncells > 0, "plan_create: empty mesh (nnodes=%lld ncells=%lld)", (long long)nnodes,
              (long long)ncells);
   FEMB_CHECK(d_dofmap && d_xdofmap, "plan_create: null dofmap");
   const int nd = elem_nd(etype);
   const int64_t nvis = ncells * nd;
   FEMB_CHECK(ncells < (int64_t(1) << 28), "plan_create: more than 2^28 cells per device is not supported");
   FEMB_CHECK(nvis < (int64_t(1) << 31) && nnodes < (int64_t(1) << 30), "plan_create: mesh too large for int32 maps");
   cudaStream_t st = as_stream(stream);

   femb200_plan *p = new femb200_plan();
   p->etype = etype, p->nd = nd, p->nv = elem_nv(etype);
   p->nnodes = nnodes, p->ncells = ncells, p->nvisits = nvis;
   p->dofmap = d_dofmap, p->xdofmap = d_xdofmap;

   int32_t *cnt = nullptr, *deg = nullptr, *flags = nullptr;
   uint32_t *tmpvis = nullptr;
   size_t scratch = 0;
   int rc = 0;
   auto fail = [&](int code) {
      cudaFree(cnt);
      cudaFree(deg);
      cudaFree(flags);
      cudaFree(tmpvis);
      femb200_plan_destroy(p);
      return code;
   };
   const int T = 256;
   if (dev_alloc(&p->nptr, (size_t)nnodes + 1, &p->bytes) || dev_alloc(&cnt, (size_t)nnodes + 1, &scratch) ||
       dev_alloc(&tmpvis, (size_t)nvis, &scratch) || dev_alloc(&flags, 2 + kNumTileR, &scratch))
      return fail(1);
   if (cudaMemsetAsync(cnt, 0, sizeof(int32_t) * ((size_t)nnodes + 1), st) != cudaSuccess ||
       cudaMemsetAsync(flags, 0, sizeof(int32_t) * (2 + kNumTileR), st) != cudaSuccess)
      return fail(set_error("plan_create: memset failed"));

   // 0. the maps come across the C ABI: refuse indices outside [0, nnodes) instead of scattering out of bounds
   k_check_range<<<(unsigned)cdiv(nvis, T), T, 0, st>>>(nvis, d_dofmap, (int32_t)nnodes, flags);
   k_check_range<<<(unsigned)cdiv(ncells * p->nv, T), T, 0, st>>>(ncells * p->nv, d_xdofmap, (int32_t)nnodes, flags);
   {
      int32_t bad = 0;
      if (cudaMemcpyAsync(&bad, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
          cudaStreamSynchronize(st) != cudaSuccess)
         return fail(set_error("plan_create: index check failed: %s", cudaGetErrorString(cudaGetLastError())));
      if (bad) return fail(set_error("plan_create: the dof map or the geometry map holds an index outside [0, %lld)", (long long)nnodes));
   }
   // 1. node -> cell visit lists
   k_count_visits<<<(unsigned)cdiv(nvis, T), T, 0, st>>>(nvis, d_dofmap, cnt);
   if ((rc = exclusive_scan_i32_i32(cnt, p->nptr, nnodes, st))) return fail(rc);
   cudaMemsetAsync(cnt, 0, sizeof(int32_t) * ((size_t)nnodes + 1), st);
   k_fill_visits<<<(unsigned)cdiv(nvis, T), T, 0, st>>>(nvis, nd, d_dofmap, p->nptr, cnt, tmpvis);
   k_sort_visits<<<(unsigned)cdiv(nnodes, T), T, 0, st>>>(nnodes, p->nptr, tmpvis);
   const bool tri = elem_is_triangle(etype);  // quadrilaterals (Q2, Q1): no fan order, natural columns, no fast records
   if (tri) k_order_visits<<<(unsigned)cdiv(nnodes, T), T, 0, st>>>(nnodes, nd, d_dofmap, p->nptr, tmpvis);

   // 2. block degrees -> brp -> bcol
   if (dev_alloc(&deg, (size_t)nnodes + 1, &scratch) || dev_alloc(&p->brp, (size_t)nnodes + 4, &p->bytes))
      return fail(1);
   k_degree<<<(unsigned)cdiv(nnodes, 128), 128, 0, st>>>(nnodes, nd, d_dofmap, p->nptr, tmpvis, deg, flags);
   if ((rc = exclusive_scan_i32_i64(deg, p->brp, nnodes, st))) return fail(rc);
   int32_t hflags[2] = {0, 0};
   if (cudaMemcpyAsync(hflags, flags, sizeof(hflags), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
       cudaMemcpyAsync(&p->nnzb, p->brp + nnodes, sizeof(int64_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
       cudaStreamSynchronize(st) != cudaSuccess)
      return fail(set_error("plan_create: pattern build failed: %s", cudaGetErrorString(cudaGetLastError())));
   if (hflags[0]) return fail(set_error("plan_create: a node has more than %d neighbour nodes", kMaxDeg));
   p->max_deg = hflags[1];
   if (dev_alloc(&p->bcol, (size_t)p->nnzb + 8, &p->bytes) || dev_alloc(&p->vrec, (size_t)nvis, &p->bytes) ||
       dev_alloc(&p->dslot, (size_t)nnodes, &p->bytes))
      return fail(1);
   k_fill_cols<<<(unsigned)cdiv(nnodes, 128), 128, 0, st>>>(nnodes, nd, d_dofmap, p->nptr, tmpvis, p->brp, p->bcol,
                                                            p->dslot);

   {  // 16-bit relative column indices for the SpMV, when every offset fits
      if (dev_alloc(&p->bcol16, (size_t)p->nnzb + 16, &p->bytes)) return fail(1);
      cudaMemsetAsync(flags, 0, sizeof(int32_t), st);
      k_cols16<<<(unsigned)cdiv(nnodes * 8, 256), 256, 0, st>>>(nnodes, p->brp, p->bcol, p->bcol16, flags);
      int32_t bad = 0;
      if (cudaMemcpyAsync(&bad, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
          cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess)
         return fail(set_error("plan_create: column offsets failed: %s", cudaGetErrorString(cudaGetLastError())));
      if (bad)
      {
         cudaFree(p->bcol16);
         p->bcol16 = nullptr;
         p->bytes -= sizeof(int16_t) * ((size_t)p->nnzb + 16);
      }
      cudaMemsetAsync(flags, 0, sizeof(int32_t) * 2, st);
   }

   // 3. slot map + staging-tile sizes
   k_fill_slots<<<(unsigned)cdiv(nnodes, 128), 128, 0, st>>>(nnodes, nd, tri, d_dofmap, p->nptr, tmpvis, p->brp, p->bcol,
                                                              p->vrec);
   {  // tile-sorted storage order (the slot map above was written node by node into a scratch copy)
      const int64_t ntiles = cdiv(nnodes, kAsmR);
      VisitRec *sorted = nullptr;
      if (dev_alloc(&sorted, (size_t)nvis, &p->bytes) || dev_alloc(&p->perm, (size_t)ntiles * kAsmR, &p->bytes) ||
          dev_alloc(&p->voff, (size_t)ntiles * kAsmLevels, &p->bytes))
         return fail(1);
      cudaMemsetAsync(flags, 0, sizeof(int32_t), st);
      k_tile_sort<<<(unsigned)ntiles, kAsmR, 0, st>>>(nnodes, p->nptr, p->vrec, sorted, p->perm, p->voff, flags);
      int32_t over = 0;
      if (cudaMemcpyAsync(&over, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
          cudaStreamSynchronize(st) != cudaSuccess)
         return fail(set_error("plan_create: tile sort failed: %s", cudaGetErrorString(cudaGetLastError())));
      cudaFree(p->vrec);
      p->bytes -= sizeof(VisitRec) * (size_t)nvis;
      p->vrec = sorted;
      if (over) return fail(set_error("plan_create: a node belongs to more than %d cells", kAsmLevels));
   }
   k_tile_max<<<(unsigned)cdiv(cdiv(nnodes, tile_r(0)), T), T, 0, st>>>(nnodes, p->brp, flags + 2);
   if (cudaMemcpyAsync(p->tile_max_blocks, flags + 2, sizeof(int32_t) * kNumTileR, cudaMemcpyDeviceToHost, st) !=
           cudaSuccess ||
       cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess)
      return fail(set_error("plan_create: slot map build failed: %s", cudaGetErrorString(cudaGetLastError())));

   // fast-path records: triangles whose kAsmR-row staging image is addressable with 15-bit byte offsets
   // and whose nodes belong to fewer than 16 cells
   if (tri && 32 * ((int64_t)p->tile_max_blocks[1] + 8) < 32768 && p->max_deg < 128)
   {
      const int64_t ntiles = cdiv(nnodes, kAsmR);
      if (dev_alloc(&p->thdr, (size_t)ntiles, &p->bytes)) return fail(1);
      cudaMemsetAsync(flags, 0, sizeof(int32_t), st);
      k_tile_hdr<<<(unsigned)cdiv(ntiles, T), T, 0, st>>>(nnodes, ntiles, p->nptr, p->brp, p->voff, p->thdr, flags);
      int32_t maxcnt = 0;
      cudaMemcpyAsync(&maxcnt, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
      if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess)
         return fail(set_error("plan_create: tile header build failed: %s", cudaGetErrorString(cudaGetLastError())));
      if (maxcnt >= 1 && maxcnt < 16)
      {
         p->flevels = maxcnt;
         const size_t nrec = (size_t)ntiles * (size_t)maxcnt * kAsmR;
         if (dev_alloc(&p->frec, nrec, &p->bytes) || dev_alloc(&p->tcnt, (size_t)ntiles * kAsmR, &p->bytes)) return fail(1);
         cudaMemsetAsync(p->frec, 0, sizeof(uint4) * nrec, st);
         cudaMemsetAsync(p->tcnt, 0, (size_t)ntiles * kAsmR, st);
         k_fast_records<<<(unsigned)ntiles, kAsmR, 0, st>>>(nnodes, nd, p->nptr, p->brp, p->perm, p->voff, p->vrec,
                                                          p->flevels, p->frec, p->tcnt);
         if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess)
            return fail(set_error("plan_create: fast record build failed: %s", cudaGetErrorString(cudaGetLastError())));
      }
   }

   cudaFree(cnt);
   cudaFree(deg);
   cudaFree(flags);
   cudaFree(tmpvis);
   *out = p;
   return 0;
}

int femb::plan_tile_cells(femb200_plan *p, int cap, cudaStream_t st)
{
   FEMB_CHECK(p && p->frec && cap > 0 && cap < 0x3ff, "plan_tile_cells: plan without fast records or bad capacity %d", cap);
   if (p->tdam_cap == cap) return 0;
   std::lock_guard<std::mutex> lock(p->range_mtx);
   if (p->tdam_cap == cap) return 0;
   FEMB_CHECK(p->tdam_cap == 0, "plan_tile_cells: the stage capacity of a plan cannot change");
   const int64_t ntiles = cdiv(p->nnodes, kAsmR);
   // tile numbers are stored in 22 bits: larger plans run without the stage (every slot = 0x3ff, no references)
   const int use_cap = ntiles < (int64_t(1) << 22) ? cap : 0;
   int32_t *crefcnt = nullptr;
   FEMB_CUDA(cudaMalloc(&p->cref, sizeof(uint32_t) * 8 * (size_t)p->ncells));
   FEMB_CUDA(cudaMalloc(&p->tdam, sizeof(int32_t) * (size_t)ntiles * (size_t)cap));
   FEMB_CUDA(cudaMalloc(&crefcnt, sizeof(int32_t) * (size_t)p->ncells));
   p->bytes += sizeof(uint32_t) * 8 * (size_t)p->ncells + sizeof(int32_t) * (size_t)ntiles * (size_t)cap;
   FEMB_CUDA(cudaMemsetAsync(p->cref, 0xff, sizeof(uint32_t) * 8 * (size_t)p->ncells, st));
   FEMB_CUDA(cudaMemsetAsync(p->tdam, 0xff, sizeof(int32_t) * (size_t)ntiles * (size_t)cap, st));
   FEMB_CUDA(cudaMemsetAsync(crefcnt, 0, sizeof(int32_t) * (size_t)p->ncells, st));
   k_tile_cells<<<(unsigned)ntiles, kAsmR, 0, st>>>(p->nnodes, p->flevels, use_cap, p->frec, p->tcnt, p->cref, crefcnt);
   const cudaError_t e1 = cudaGetLastError(), e2 = cudaStreamSynchronize(st);
   cudaFree(crefcnt);
   FEMB_CHECK(e1 == cudaSuccess && e2 == cudaSuccess, "plan_tile_cells: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
   p->tdam_cap = cap;
   p->tdam_refs = use_cap > 0;
   return 0;
}

extern "C" int femb200_plan_sizes(const femb200_plan *p, int64_t *nnodes, int64_t *ncells, int64_t *nnz_blocks,
                                  int64_t *nnz, int32_t *max_block_degree, int64_t *device_bytes)
{
   FEMB_CHECK(p != nullptr, "plan_sizes: null plan");
   if (nnodes) *nnodes = p->nnodes;
   if (ncells) *ncells = p->ncells;
   if (nnz_blocks) *nnz_blocks = p->nnzb;
   if (nnz) *nnz = 4 * p->nnzb;
   if (max_block_degree) *max_block_degree = p->max_deg;
   if (device_bytes) *device_bytes = (int64_t)p->bytes;
   return 0;
}

extern "C" int femb200_plan_block_csr(const femb200_plan *p, const int64_t **d_brp, const int32_t **d_bcol)
{
   FEMB_CHECK(p != nullptr, "plan_block_csr: null plan");
   if (d_brp) *d_brp = p->brp;
   if (d_bcol) *d_bcol = p->bcol;
   return 0;
}

extern "C" int femb200_plan_copy_block_csr(const femb200_plan *p, int64_t *d_brp, int32_t *d_bcol, void *stream)
{
   FEMB_CHECK(p && d_brp && d_bcol, "plan_copy_block_csr: null argument");
   cudaStream_t st = as_stream(stream);
   FEMB_CUDA(cudaMemcpyAsync(d_brp, p->brp, sizeof(int64_t) * (size_t)(p->nnodes + 1), cudaMemcpyDeviceToDevice, st));
   FEMB_CUDA(cudaMemcpyAsync(d_bcol, p->bcol, sizeof(int32_t) * (size_t)p->nnzb, cudaMemcpyDeviceToDevice, st));
   return 0;
}

extern "C" int femb200_plan_scalar_csr(const femb200_plan *p, int64_t *d_rowptr, int32_t *d_colidx, void *stream)
{
   FEMB_CHECK(p && d_rowptr && d_colidx, "plan_scalar_csr: null argument");
   const int T = 256;
   k_scalar_csr<<<(unsigned)cdiv(p->nnodes * 32, T), T, 0, as_stream(stream)>>>(p->nnodes, p->brp, p->bcol, d_rowptr,
                                                                               d_colidx);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_plan_set_dirichlet(femb200_plan *p, const uint8_t *d_bc, void *stream)
{
   FEMB_CHECK(p != nullptr, "plan_set_dirichlet: null plan");
   cudaStream_t st = as_stream(stream);
   cudaFree(p->norm_partials);
   p->norm_partials = nullptr;
   cudaFree(p->bc_nodes);
   p->bc_nodes = nullptr;
   p->nbc = 0;
   cudaFree(p->lift_nodes);
   p->lift_nodes = nullptr;
   p->nlift = 0;
   if (!d_bc)
   {
      cudaFree(p->bc);
      p->bc = nullptr;
      return 0;
   }
   size_t acc = 0;
   if (!p->bc && dev_alloc(&p->bc, (size_t)(2 * p->nnodes), &acc)) return 1;
   FEMB_CUDA(cudaMemcpyAsync(p->bc, d_bc, (size_t)(2 * p->nnodes), cudaMemcpyDeviceToDevice, st));
   int32_t *count = nullptr;
   if (dev_alloc(&count, 1, &acc)) return 1;
   const int T = 256;
   cudaMemsetAsync(count, 0, sizeof(int32_t), st);
   k_bc_nodes<<<(unsigned)cdiv(p->nnodes, T), T, 0, st>>>(p->nnodes, p->bc, nullptr, count);
   int32_t n = 0;
   cudaMemcpyAsync(&n, count, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
   if (cudaStreamSynchronize(st) != cudaSuccess)
   {
      cudaFree(count);
      return set_error("plan_set_dirichlet: %s", cudaGetErrorString(cudaGetLastError()));
   }
   if (dev_alloc(&p->bc_nodes, (size_t)n, &acc))
   {
      cudaFree(count);
      return 1;
   }
   cudaMemsetAsync(count, 0, sizeof(int32_t), st);
   k_bc_nodes<<<(unsigned)cdiv(p->nnodes, T), T, 0, st>>>(p->nnodes, p->bc, p->bc_nodes, count);
   p->nbc = n;
   // the node rows apply_lifting touches: every row with a constrained column (the constrained nodes among them)
   uint8_t *mark = nullptr;
   int32_t nl = 0;
   if (n > 0)
   {
      if (dev_alloc(&mark, (size_t)p->nnodes, &acc))
      {
         cudaFree(count);
         return 1;
      }
      cudaMemsetAsync(mark, 0, (size_t)p->nnodes, st);
      k_mark_lift_rows<<<(unsigned)cdiv((int64_t)n * 32, T), T, 0, st>>>(n, p->bc_nodes, p->brp, p->bcol, mark);
      cudaMemsetAsync(count, 0, sizeof(int32_t), st);
      k_compact_marked<<<(unsigned)cdiv(p->nnodes, T), T, 0, st>>>(p->nnodes, mark, nullptr, count);
      cudaMemcpyAsync(&nl, count, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
      if (cudaStreamSynchronize(st) != cudaSuccess || dev_alloc(&p->lift_nodes, (size_t)nl, &acc))
      {
         cudaFree(count), cudaFree(mark);
         return set_error("plan_set_dirichlet: lifting rows: %s", cudaGetErrorString(cudaGetLastError()));
      }
      cudaMemsetAsync(count, 0, sizeof(int32_t), st);
      k_compact_marked<<<(unsigned)cdiv(p->nnodes, T), T, 0, st>>>(p->nnodes, mark, p->lift_nodes, count);
   }
   cudaStreamSynchronize(st);
   cudaFree(count);
   cudaFree(mark);
   p->nlift = nl;
   FEMB_LAUNCH_CHECK();
   return 0;
}

namespace femb {
// SpMV tiling of the node rows [lo, hi): the bulk-copy staged kernel sizes its shared-memory stages for the
// largest tile.  Ranges that start on a 64-row boundary share the plan's aligned tiles; any other range (the
// owned rows of a rank) is measured once (synchronises the device) and cached in the plan.
int plan_row_range(const femb200_plan *p, int64_t lo, int64_t hi, RowRange *out)
{
   FEMB_CHECK(p != nullptr, "row range: null plan");
   FEMB_CHECK(0 <= lo && lo <= hi && hi <= p->nnodes, "row range: bad range [%lld, %lld) of %lld node rows", (long long)lo,
              (long long)hi, (long long)p->nnodes);
   out->lo = lo, out->hi = hi;
   out->tile_max[0] = p->tile_max_blocks[0], out->tile_max[1] = p->tile_max_blocks[1];
   if (lo % 64 == 0 || hi == lo) return 0;
   femb200_plan *pm = const_cast<femb200_plan *>(p);
   std::lock_guard<std::mutex> lock(pm->range_mtx);
   auto it = pm->range_tile_max.find(std::make_pair(lo, hi));
   if (it == pm->range_tile_max.end())
   {
      int32_t *d = nullptr, h[2] = {0, 0};
      FEMB_CUDA(cudaMalloc(&d, 2 * sizeof(int32_t)));
      FEMB_CUDA(cudaMemset(d, 0, 2 * sizeof(int32_t)));
      for (int k = 0; k < 2; ++k)
      {
         const int R = 32 << k;
         const int64_t nt = cdiv(hi - lo, R);
         k_range_tile_max<<<(unsigned)cdiv(nt, 256), 256>>>(lo, hi, R, p->brp, d + k);
      }
      const cudaError_t e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
      cudaFree(d);
      FEMB_CHECK(e == cudaSuccess, "row range: %s", cudaGetErrorString(e));
      it = pm->range_tile_max.emplace(std::make_pair(lo, hi), std::array<int32_t, 2>{h[0], h[1]}).first;
   }
   out->tile_max[0] = it->second[0], out->tile_max[1] = it->second[1];
   return 0;
}
}  // namespace femb

namespace femb {
int plan_cell_scratch(femb200_plan *p)
{
   if (p->celld) return 0;
   std::lock_guard<std::mutex> lock(p->range_mtx);
   if (p->celld) return 0;
   const size_t bytes = sizeof(double) * plan_cell_scratch_doubles(p->etype) * (size_t)p->ncells;
   FEMB_CUDA(cudaMalloc(&p->celld, bytes));
   p->bytes += bytes;
   return 0;
}
}  // namespace femb

extern "C" int femb200_plan_set_option(femb200_plan *p, const char *key, int value)
{
   FEMB_CHECK(p && key, "plan_set_option: null argument");
   if (!strcmp(key, "assembly_path"))
   {
      FEMB_CHECK(value >= 0 && value <= 2, "plan_set_option: assembly_path must be 0 (auto), 1 (visit records) or 2 (per point)");
      p->opt_assembly_path = value;
   }
   else if (!strcmp(key, "damage_stage"))
   {
      FEMB_CHECK(value >= 0 && value <= 2, "plan_set_option: damage_stage must be 0 (auto), 1 (always) or 2 (never)");
      p->opt_dmg_stage = value;
   }
   else if (!strcmp(key, "spmv_path"))
   {
      FEMB_CHECK(value == 0 || value == 1, "plan_set_option: spmv_path must be 0 (auto) or 1 (direct)");
      p->opt_spmv_path = value;
   }
   else if (!strcmp(key, "spmv_cols"))
   {
      FEMB_CHECK(value == 0 || value == 1, "plan_set_option: spmv_cols must be 0 (auto: 16-bit relative indices) or 1 (32-bit)");
      p->opt_spmv_cols = value;
   }
   else if (!strcmp(key, "vector_path"))
   {
      FEMB_CHECK(value == 0 || value == 1, "plan_set_option: vector_path must be 0 (two passes) or 1 (single-pass gather)");
      p->opt_vector_path = value;
   }
   else if (!strcmp(key, "prefetch_tiles"))
      p->opt_prefetch_tiles = value;
   else if (!strcmp(key, "stream_out"))
   {
      FEMB_CHECK(value == 0 || value == 1, "plan_set_option: stream_out must be 0 (auto: tensor bulk stores) or 1 (store loop)");
      p->opt_stream_out = value;
   }

   else
      return set_error("plan_set_option: unknown key '%s'", key);
   return 0;
}

extern "C" int femb200_plan_get_option(const femb200_plan *p, const char *key, int *value)
{
   FEMB_CHECK(p && key && value, "plan_get_option: null argument");
   if (!strcmp(key, "assembly_path"))
      *value = p->opt_assembly_path;
   else if (!strcmp(key, "damage_stage"))
      *value = p->opt_dmg_stage;
   else if (!strcmp(key, "spmv_path"))
      *value = p->opt_spmv_path;
   else if (!strcmp(key, "spmv_cols"))
      *value = p->opt_spmv_cols;
   else if (!strcmp(key, "vector_path"))
      *value = p->opt_vector_path;
   else if (!strcmp(key, "prefetch_tiles"))
      *value = p->opt_prefetch_tiles;
   else if (!strcmp(key, "stream_out"))
      *value = p->opt_stream_out;
   else if (!strcmp(key, "spmv_col_bits"))
      *value = (p->bcol16 && p->opt_spmv_cols != 1) ? 16 : 32;
   else if (!strcmp(key, "fast_records"))
      *value = p->frec ? 1 : 0;
   else
      return set_error("plan_get_option: unknown key '%s'", key);
   return 0;
}
