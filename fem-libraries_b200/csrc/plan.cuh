// plan.cuh -- the assembly plan: node->cell visit lists, node-block CSR pattern and
// the per-visit slot map of the write-once gather assembly.
#pragma once
#include <array>
#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

namespace femb {

constexpr int kAsmLevelsFwd = 16;  // = kAsmLevels (declared below)

// One visit = (row node I, incident cell e, local index a of I in e).  16 bytes:
//   word 0   cell id e
//   word 1   a (bits 0-7) | slot of local dof 8 (bits 8-15, Q2 only) | first-touch mask (bits 16-31):
//            bit b set when this visit is the first (in list order) to contribute to
//            slot[b], so it stores instead of adds
//   word 2-3 slot in block row I of the column stored at position t = 0..7, one byte each; triangles
//            store the columns in ROTATED order (position t = local dof (m + t) mod 3 for the vertices,
//            3 + (m + t - 3) mod 3 for the edges, m = a mod 3: the row's own vertex / edge comes first),
//            quadrilaterals in natural order; the first-touch bits use the same positions
// nptr[I] .. nptr[I+1] counts the visits of node I (ascending cell id: the order of the sums).
// STORAGE ORDER of vrec: tiles of kAsmR consecutive nodes; inside a tile the nodes are ranked by
// decreasing visit count (perm[n0 + rank] = tile-local node) and the records are laid out level by
// level: record (rank r, visit j) lives at nptr[n0] + voff[tile][j] + r, so the lanes of a warp
// (consecutive ranks, same j) read consecutive 16-byte records.
struct __align__(16) VisitRec
{
   uint32_t e;
   uint8_t a;
   uint8_t slot8;
   uint16_t first;
   uint8_t slot[8];
};
// register-friendly decoded form
struct Visit
{
   uint32_t e, a, first, slot8;
   uint64_t slots;
   __device__ __forceinline__ explicit Visit(const uint4 raw)
       : e(raw.x), a(raw.y & 0xffu), first(raw.y >> 16), slot8((raw.y >> 8) & 0xffu),
         slots((uint64_t)raw.z | ((uint64_t)raw.w << 32))
   {
   }
   __device__ __forceinline__ int slot(int b) const { return b < 8 ? (int)((slots >> (8 * b)) & 0xffu) : (int)slot8; }
   __device__ __forceinline__ bool is_first(int b) const { return (first >> b) & 1u; }
};
static_assert(sizeof(VisitRec) == 16, "VisitRec must be 16 bytes");

// staging swizzle on 16-byte units: spreads the systematically aligned row starts of neighbouring
// threads over different bank groups; an involution inside aligned groups of 8 units, so the
// stream-out stays coalesced.  key = bit-reversed low 3 bits of the aligned 8-unit group index
// (chosen by simulating the staging accesses of P1 / P2 tiles: fewest shared-memory wavefronts)
__host__ __device__ __forceinline__ int swz(int u)
{
   const int g = u >> 3;
   return u ^ (((g & 1) << 2) | (g & 2) | ((g >> 2) & 1));
}

// Staging layout of the FAST kernel (round 2).  Position p = (first 16-byte unit of the tile in the value array mod 8)
// + tile-local unit: the 128-byte lines of the image coincide with the 128-byte lines of the value array, and the
// 16-byte chunk inside a line is XORed with the line index mod 8.  That is the TMA SWIZZLE_128B pattern (byte address
// bits [4:6] ^= bits [7:9], image base 1024-byte aligned): the finished tile leaves with tensor bulk stores
// (cp.async.bulk.tensor, UTMASTG) which undo the swizzle on the way out, instead of an LDS + STG loop over 30 KB.
// (The simulated conflict factor of this key is 1.56 against 1.34 for the bit-reversed one of swz(): about 4 % more
// staging wavefronts, against a quarter of the kernel's LSU wavefronts saved.)
__host__ __device__ __forceinline__ int swz_tma(int p) { return p ^ ((p >> 3) & 7); }

// Fast-path record of one visit, triangles only: everything the two row threads of the node (scalar rows h = 0, 1)
// need in one 16-byte load (both load the same address), with the staging positions resolved at plan time:
//   x   cell id e (bits 0-27) | number of visits of the row (bits 28-31; cells are numbered below 2^28)
//   y   position of column 0 (bits 0-10) | column 1 (11-21) | first-touch bits of the five puts (22-26) | carry-out (27)
//       | edge row (28) | local vertex number of the visit's vertex 1' (29-30)
//   z   position of column 2 (0-10) | column 3 (11-21) | block degree of the node (22-28) | local vertex number of 2' (29-30)
//   w   position of column 4 (0-10) | column 5 (11-21) | slot of the cell in the tile's damage-record stage (22-31;
//       0x3ff: not staged; written by plan_tile_cells on the first damaged assembly)
// "Position" = 16-byte unit of the column in the tile image for scalar row 0, BEFORE the chunk swizzle (swz_tma above),
// columns in rotated order as in VisitRec (t = 0..5); the row-1 thread adds the block degree (its row follows row 0 in
// the CSR) and both apply the swizzle (three integer operations).  The five puts are positions 1..5 of a vertex row,
// 0, 1, 2, 4, 5 of an edge row (the diagonal block never goes through the image before its final store).  Put / carry /
// flip semantics: k_fast_records.  One record per visit instead of one per (visit, scalar row) halves the largest
// read stream of the kernel (0.8 -> 0.4 GB at n = 1448).
// Storage: fixed stride, record (tile, level j, rank r) at (tile * flevels + j) * kAsmR + r with flevels = the largest
// visit count of the mesh (zero padding where a row has fewer visits): the address depends on the block and thread index
// only, and the 16 ranks of a warp read 256 contiguous bytes.
// Per-tile header of the streaming assembly kernel: everything a CTA needs to know about a tile in
// one 64-byte bulk copy.
struct __align__(64) TileHdr
{
   int64_t b0;                  // first node block of the tile (brp[n0])
   int32_t vbase, nvis, units;  // first visit record, number of visits, 16-byte units of the tile image
   int32_t pad;
   uint16_t voff[kAsmLevelsFwd];  // level offsets (records in levels < j)
   uint16_t pad2[4];
};
constexpr int kAsmR = 64;      // node rows per assembly tile (fixed at plan time: vrec storage order)
constexpr int kAsmLevels = 16; // visits per node supported by the tile-sorted layout
static_assert(kAsmLevels == kAsmLevelsFwd, "TileHdr::voff");
static_assert(sizeof(TileHdr) == 64, "TileHdr must be 64 bytes");
constexpr int kNumTileR = 6;
// Stencil dictionary of the SpMV (spmv.cu): the distinct lists of column offsets J - I of the node rows, at most
// kStencilK lists of at most kStencilD offsets (a lattice numbering has a handful: 16 for P2 triangles).
constexpr int kStencilK = 64;
constexpr int kStencilD = 32;
// Compact values of the PCG (P2 triangles with a stencil dictionary): the blocks of a vertex and the midpoint of the
// opposite edge are zero on every straight-sided cell (their gradient products integrate (4 l_a - 1) l_b to 0), and no
// other cell holds that pair.  A compact key = (stencil id, mask of the kept slots); its dictionary entry holds, in
// int16 words: the stencil's column offsets [kStencilD], the degree, the kept degree, and per slot its position in the
// compact row or -1 when the block is dropped [kStencilD].  33 words per entry: keys start in different banks.
constexpr int kCompactK = 64;
constexpr int kCDictStride = 2 * kStencilD + 2;
__host__ __device__ constexpr int tile_r(int r) { return r == 0 ? 32 : r == 1 ? 64 : r == 2 ? 96 : r == 3 ? 128 : r == 4 ? 192 : 256; }

}  // namespace femb

struct femb200_plan
{
   int etype = 0, nd = 0, nv = 0;
   int64_t nnodes = 0, ncells = 0, nnzb = 0, nvisits = 0;
   int32_t max_deg = 0;
   const int32_t *dofmap = nullptr, *xdofmap = nullptr;  // borrowed
   int32_t *nptr = nullptr;                               // [nnodes+1]
   femb::VisitRec *vrec = nullptr;                        // [nvisits], tile-sorted (see above)
   uint4 *frec = nullptr;                                 // [ntiles * flevels * kAsmR] fast-path records (triangles) or null
   uint8_t *tcnt = nullptr;                               // [ntiles * kAsmR] visit count of (tile, rank) (with frec)
   femb::TileHdr *thdr = nullptr;                         // [ntiles] tile headers (with frec)
   int32_t flevels = 0;                                   // levels of the fixed-stride frec layout (max visits per node)
   uint8_t *perm = nullptr;                               // [ntiles * kAsmR] rank -> tile-local node
   uint16_t *voff = nullptr;                              // [ntiles * kAsmLevels] level offsets in a tile
   int64_t *brp = nullptr;                                // [nnodes+1]
   int32_t *bcol = nullptr;                               // [nnzb]
   int16_t *bcol16 = nullptr;                             // [nnzb] bcol[k] - (node of the row), or null when one does not fit
   // stencil ids (null / 0 when the pattern has no dictionary): row I's bcol16 list is stencil_off[sig[I]][0, deg)
   uint8_t *sig = nullptr;                                // [nnodes] stencil id of each node row
   int16_t *stencil_off = nullptr;                        // [nstencils][kStencilD] offsets, in the plan's column order
   uint8_t *stencil_deg = nullptr;                        // [nstencils] block degree of each stencil
   int32_t nstencils = 0;
   // compact values of the PCG (plan.cuh above; null / 0 when the plan has none): the kept blocks of row I are
   // cvalues[4 cbrp[I], 4 cbrp[I + 1]) in the scalar-row layout of the CSR (kept row-0 halves, then row-1 halves)
   uint8_t *csig = nullptr;        // [nnodes] compact key of each node row
   int16_t *cdict = nullptr;       // [ncompact][kCDictStride]
   int64_t *cbrp = nullptr;        // [nnodes+1] first kept block of each node row
   int32_t ncompact = 0;
   int64_t nkept = 0;
   int32_t ctile_max = 0;          // kept blocks of the largest 64-row tile (tiles aligned to 64 rows)
   double *cvalues = nullptr;      // [4 nkept] allocated by the first solve that uses it (cg.cu), then kept
   int *cbad = nullptr;            // device word: set by a solve's first apply when a dropped block is not +-0
   bool cvalues_failed = false;    // the allocation failed once: solves take the full path
   uint8_t *dslot = nullptr;                              // [nnodes] slot of the diagonal block in its row (255: none)
   int32_t tile_max_blocks[femb::kNumTileR] = {0, 0, 0, 0, 0, 0};
   // Dirichlet
   uint8_t *bc = nullptr;        // [2*nnodes] or null
   int32_t *bc_nodes = nullptr;  // compact list of constrained nodes
   int32_t nbc = 0;
   int32_t *lift_nodes = nullptr;  // compact list of the node rows with a constrained column (the rows apply_lifting changes)
   int32_t nlift = 0;
   double *norm_partials = nullptr;  // [3 nbc] scratch of femb200_assemble_matrix_norms
   size_t bytes = 0;
   double *celld = nullptr;    // damage records of the cells (assemble.cu, cell_setup_damage_kernel), lazily allocated
   int32_t *celld_count = nullptr;  // [1 + ncells]: number of damaged cells, then their list
   // damage-record stage of the fast kernel (plan_tile_cells, built on the first damaged assembly): every distinct cell
   // of a tile has a slot in the tile's stage (number in the fast records); cref[cell] = up to 6 x (tile << 10 | slot),
   // slot 0x3ff: visited but not staged, 0xffffffff: unused; tdam[tile][slot] = the cell when it is damaged in the current assembly, else -1
   uint32_t *cref = nullptr;   // [ncells][8]
   int32_t *tdam = nullptr;    // [ntiles][tdam_cap]
   // damaged cells of the last damaged assembly: device counter (pre-pass), host-mapped word (and its device address)
   int *dmg_counter = nullptr, *dmg_count = nullptr, *dmg_count_dev = nullptr;
   int opt_dmg_stage = 0;      // 0 auto (by the share of damaged cells of the previous assembly), 1 always, 2 never
   int32_t tdam_cap = 0;
   bool tdam_refs = false;     // cref is filled (false: more than 2^22 tiles, no stage)
   double *cellrec = nullptr;  // [ncells][4] per-cell sqrt(|T| E) (grad l1, grad l2), fast path, lazily allocated
   // tensor maps of the value array the fast kernel last wrote (boxes of 8 lines and of 1 line of 128 bytes)
   alignas(64) unsigned char tmap[2][128] = {};
   const void *tmap_values = nullptr;
   int opt_stream_out = 0;  // 0 auto (tensor bulk stores when available), 1 LDS + STG loop
   // Kernel selection of this plan (femb200_plan_set_option): the fallback kernels that serve plans without
   // fast records / oversized SpMV tiles can be forced, so that the tests cover them on any mesh.
   int opt_assembly_path = 0;    // 0 auto; 1 visit-record kernel; 2 per-quadrature-point kernel
   int opt_spmv_path = 0;        // 0 auto (bulk-copy staged, persistent); 1 direct kernel
   int opt_spmv_cols = 0;        // 0 auto (stencil ids, else 16-bit relative indices, else 32-bit); 1 32-bit; 2 16-bit
   int opt_spmv_compact = 0;     // 0 auto (PCG applies stream the compact values when the plan has them); 1 off
   int opt_vector_path = 0;      // residual vector: 0 two passes (per-cell r_e + gather); 1 single-pass gather
   int opt_prefetch_tiles = -1;  // record prefetch distance of the assembly kernel in tiles (-1: 8 x SM count)
   // largest 32- / 64-row SpMV tile (in node blocks) of the tiling that starts at row_lo, then the largest 64-row tile
   // of the compact values, per row range [row_lo, row_hi) that has been applied (the owned rows of a rank; measured
   // once, on first use)
   std::map<std::pair<int64_t, int64_t>, std::array<int32_t, 3>> range_tile_max;
   std::mutex range_mtx;
};

namespace femb {
// [lo, hi) = node rows to apply; tile_max from plan_range_tile_max()
struct RowRange
{
   int64_t lo, hi;
   int32_t tile_max[2];
   int32_t ctile_max;  // largest 64-row tile of the compact values (0: the plan has none)
};
// builds p->cref / allocates p->tdam for a record stage of `cap` cells per tile and writes the slot numbers into the
// fast records
int plan_tile_cells(femb200_plan *p, int cap, cudaStream_t st);
int plan_row_range(const femb200_plan *p, int64_t lo, int64_t hi, RowRange *out);
// doubles per cell of the plan's per-cell scratch p->celld: the damage records of the matrix assembly (P1: 96-byte
// slots, P2: 192-byte slots) and the element vectors of the residual assembly (2 nd doubles: 6 / 12 / 18)
inline size_t plan_cell_scratch_doubles(int etype) { return etype == FEMB200_P1 ? 12 : 24; }
// allocates p->celld on first use
int plan_cell_scratch(femb200_plan *p);
// compact: 0 the CSR values; 1 the CSR values, and the kept blocks are written to p->cvalues (a dropped block that is
// not +-0 sets *p->cbad); 2 the compact values when *p->cbad == 0, else the CSR values (switched on the device).
int spmv_launch(const femb200_plan *p, const RowRange &rr, const double *d_values, const double *d_x, double *d_y,
                const double *d_flag, double *d_dot_out, bool accumulate, cudaStream_t st, int compact = 0);
// true when the PCG applies of rr can use the compact values (option, plan, stage sizes); allocates p->cvalues and
// p->cbad on first use and returns false when that fails
bool spmv_compact_ready(femb200_plan *p, const RowRange &rr);
}  // namespace femb
