// dist.cuh -- shared declarations of the multi-GPU layer (dist.cu) and the PCG loop (cg.cu).
//
// Role in the reference: the MPI layer under the linear solve -- the forward ghost update before an
// operator apply (VecGhostUpdate(INSERT, FORWARD), F.cc:865-866; the halo inside HypreParMatrix::Mult)
// and the MPI_Allreduce of the CG dot products inside mfem::CGSolver / PETSc KSP cg (M.cc:1502-1528,
// F.cc:718-722).
//
// B200 design: one process per GPU.  Two transports behind the same entry points:
//  * P2P (default on one NVSwitch box): every rank owns an ARENA (one cudaMalloc: header + the CG work
//    vectors) exported with a CUDA IPC handle and mapped by all peers.  The halo is a kernel that STORES
//    the interface rows of the search direction straight into the neighbours' ghost rows over NVLink,
//    signals a sequence-numbered flag and waits for the neighbours' flags; the all-reduce of a CG dot
//    product is fused into the one-warp scalar kernel that follows every dot: lane p stores this rank's
//    partial into rank p's mailbox and polls its own mailbox p, the warp sums the world partials in rank
//    order (bit-identical on every rank).  No NCCL launch, no host involvement; sequence numbers live in
//    device memory, so a captured CUDA graph of one CG iteration can be replayed.
//  * NCCL (any ncclComm_t of the same size): grouped ncclSend/ncclRecv + ncclAllReduce of one double,
//    enqueued on the caller's stream (also graph-captured).  The baseline the P2P transport is measured
//    against, and the path for communicators that span nodes.
#pragma once
#include "plan.cuh"

namespace femb {

constexpr int kMaxWorld = 16;  // ranks of one job (lanes of the scalar warp)
constexpr int kMaxNeigh = 8;   // halo neighbours of a rank
constexpr int kRedSets = 4;    // mailbox sets, used round robin (a rank is never more than one reduction ahead)
constexpr int kRedVals = 3;    // doubles per mailbox message

struct RedSlot
{
   double v[kRedVals];
   unsigned long long flag;  // sequence number of the message in v
};

// First bytes of every rank's arena.  Written by the peers (red, halo_flag) and by this rank's own
// one-thread epilogues (the sequence counters).
struct ArenaHdr
{
   RedSlot red[kRedSets][kMaxWorld];         // [set][sender rank]
   unsigned long long halo_flag[kMaxWorld];  // [sender rank]: sequence number of the last halo it delivered
   unsigned long long seq_red, seq_halo;     // this rank's counters
   unsigned int halo_ticket;
   int error;                                // set when a wait timed out (peer died / mismatched call sequence)
};
constexpr size_t kArenaHdrBytes = 4096;
static_assert(sizeof(ArenaHdr) <= kArenaHdrBytes, "arena header");

// by-value kernel argument of the fused all-reduce
struct RedArgs
{
   int world = 1, rank = 0;
   ArenaHdr *hdr = nullptr;  // null: no mailbox all-reduce (single rank, or the NCCL transport did it already)
   ArenaHdr *peer[kMaxWorld] = {};
};

}  // namespace femb

struct femb200_dist;

namespace femb {

// the operator and vectors of one PCG solve (local numbering: owned rows [own_lo, own_hi), ghosts around)
struct CgProblem
{
   const femb200_plan *plan = nullptr;
   int op_kind = 0;
   const void *op = nullptr;
   const double *values = nullptr;
   int64_t own_lo = 0, own_hi = 0;
   const double *b = nullptr, *dinv = nullptr;
   double *x = nullptr;
   double *r = nullptr, *d = nullptr, *z = nullptr, *scal = nullptr;
   double rtol = 1e-12, atol = 0.;
   int maxit = 0, check_every = 25, fixed_iters = 0;
   femb200_dist *comm = nullptr;  // null: single GPU
   bool use_graph = false;
};
int cg_core(const CgProblem &P, int *iters, double *final_norm, int *converged, cudaStream_t st);

// hooks implemented in dist.cu (all no-ops for a null / single-rank comm)
RedArgs dist_red_args(femb200_dist *D);
int dist_allreduce_pre(femb200_dist *D, double *d_val, int count, cudaStream_t st);  // NCCL transport: enqueue the all-reduce
int dist_halo_arena(femb200_dist *D, cudaStream_t st);  // ghost update of the arena's search direction
int dist_check_error(femb200_dist *D, cudaStream_t st);

// one cached CUDA graph of a full CG iteration
struct IterGraph
{
   cudaGraphExec_t exec = nullptr;
   const void *key[8] = {};
   int64_t ikey[4] = {};
};
IterGraph *dist_iter_graph(femb200_dist *D);
cudaStream_t dist_capture_stream(femb200_dist *D);

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p)
{
   unsigned long long v;
   asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
   return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v)
{
   asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_f64(double *p, double v)
{
   asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double *p)
{
   double v;
   asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
   return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
   unsigned long long t;
   asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
   return t;
}
constexpr unsigned long long kWaitTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;  // 20 s: a peer is gone

// All-reduce (sum) of up to kRedVals doubles over the ranks, by ONE WARP (lane p talks to rank p).
// Every lane passes the same `mine`; every lane returns the same sums, added in rank order.
template <int NV>
__device__ __forceinline__ void mailbox_allreduce(const RedArgs &ra, double (&mine)[NV])
{
   static_assert(NV <= kRedVals, "mailbox message size");
   const int lane = threadIdx.x & 31;
   ArenaHdr *hdr = ra.hdr;
   const unsigned long long seq = hdr->seq_red + 1;
   const int set = (int)(seq & (kRedSets - 1));
   __syncwarp();  // every lane has read seq_red before lane 0 advances it
   double v[NV];
#pragma unroll
   for (int k = 0; k < NV; ++k) v[k] = 0.;
   if (lane < ra.world)
   {
      RedSlot *out = &ra.peer[lane]->red[set][ra.rank];
#pragma unroll
      for (int k = 0; k < NV; ++k) st_relaxed_sys_f64(&out->v[k], mine[k]);
      st_release_sys_u64(&out->flag, seq);  // release: the payload is visible before the flag
      const RedSlot *in = &hdr->red[set][lane];
      const unsigned long long t0 = global_timer_ns();
      while (ld_acquire_sys_u64(&in->flag) < seq)
         if (global_timer_ns() - t0 > kWaitTimeoutNs)
         {
            hdr->error = 1;
            break;
         }
#pragma unroll
      for (int k = 0; k < NV; ++k) v[k] = ld_relaxed_sys_f64(&in->v[k]);
   }
#pragma unroll
   for (int k = 0; k < NV; ++k)
   {
      double s = 0.;
      for (int p = 0; p < ra.world; ++p) s += __shfl_sync(0xffffffffu, v[k], p);
      mine[k] = s;
   }
   __syncwarp();
   if (lane == 0) hdr->seq_red = seq;
}

}  // namespace femb
