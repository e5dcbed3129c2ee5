// cg.cu -- (Jacobi-)preconditioned conjugate gradients with device-resident
// scalars.
//
// Role in the reference: mfem::CGSolver lin_solv (SetRelTol 1e-12, SetMaxIter
// 2000, M.cc:1502,1525-1528) / PETSc KSP cg (F.cc:718-722) called by the Newton
// solver once per non-linear iteration.  The reference preconditions with HYPRE
// BoomerAMG (third party, out of scope: SURVEY.md 2 #6); here B = diag(A)^-1 or I.
//
// Semantics are mfem::CGSolver::Mult's: zero initial guess, r = b, d = B r,
// nom = <d, r>, r0 = max(nom rtol^2, atol^2); per iteration
//    alpha = nom / den;  x += alpha d;  r -= alpha A d;  betanom = <B r, r>;
//    stop if betanom <= r0;  beta = betanom / nom;  d = B r + beta d;
//    den = <d, A d>;  nom = betanom.
// One iteration is 3 vector kernels (update_r, update_xdir, spmv+dot: x += alpha d rides with the direction update, which
// reads d anyway -- 10 vector passes instead of 11 next to the operator apply) and 2
// one-thread scalar kernels; the host never reads a scalar inside the loop except
// for the convergence poll every `check_every` iterations.  After convergence the
// remaining queued kernels see flag != 0 and return immediately.
//
// The multi-GPU driver (femb200/dist.py) calls the same kernels one by one and
// all-reduces the freshly written partial (scal[SC_RED_*]) between a vector
// kernel and its scalar kernel: the analogue of the MPI_Allreduce inside
// CGSolver / KSP.
#include <algorithm>

#include "cg_slots.cuh"
#include "dist.cuh"
#include "reduce.cuh"

namespace femb {

int pa_apply_launch(const femb200_pa *pa, const double *d_x, double *d_y, const double *d_flag, double *d_dot_out,
                    cudaStream_t st, bool accumulate);
}  // namespace femb
int64_t pa_num_dofs(const femb200_pa *pa);
namespace femb {

constexpr int kVecThreads = 256;

// x = 0, r = b, d = B b, partial <d, r>
__global__ void __launch_bounds__(kVecThreads)
cg_init_kernel(int64_t n, const double *__restrict__ b, const double *__restrict__ dinv, double *__restrict__ x,
               double *__restrict__ r, double *__restrict__ d, ReduceScratch red, double *__restrict__ out)
{
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n; i += stride)
   {
      const double bi = b[i];
      const double di = dinv ? dinv[i] * bi : bi;
      x[i] = 0.;
      r[i] = bi;
      d[i] = di;
      part += di * bi;
   }
   block_reduce_finish<kVecThreads>(part, red, out);
}

// x += alpha d;  r -= alpha z;  partial <B r, r>
__global__ void __launch_bounds__(kVecThreads)
cg_update_xr_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ d,
                    const double2 *__restrict__ z, const double2 *__restrict__ dinv, double2 *__restrict__ x,
                    double2 *__restrict__ r, ReduceScratch red, double *__restrict__ out)
{
   if (scal[SC_FLAG] != 0.) return;
   const double alpha = scal[SC_NOM] / scal[SC_DEN];
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 di = d[i], zi = z[i];
      double2 xi = x[i], ri = r[i];
      xi.x = __fma_rn(alpha, di.x, xi.x), xi.y = __fma_rn(alpha, di.y, xi.y);
      ri.x = __fma_rn(-alpha, zi.x, ri.x), ri.y = __fma_rn(-alpha, zi.y, ri.y);
      x[i] = xi;
      r[i] = ri;
      if (dinv)
      {
         const double2 pi = dinv[i];
         part = __fma_rn(__dmul_rn(pi.x, ri.x), ri.x, part), part = __fma_rn(__dmul_rn(pi.y, ri.y), ri.y, part);
      }
      else
         part = __fma_rn(ri.x, ri.x, part), part = __fma_rn(ri.y, ri.y, part);
   }
   block_reduce_finish<kVecThreads>(part, red, out);
}

// d = B r + beta d
__global__ void __launch_bounds__(kVecThreads)
cg_update_dir_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ r,
                     const double2 *__restrict__ dinv, double2 *__restrict__ d)
{
   if (scal[SC_FLAG] != 0.) return;
   const double beta = scal[SC_BETA];
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n2; i += stride)
   {
      double2 ri = r[i];
      if (dinv)
      {
         const double2 pi = dinv[i];
         ri.x = __dmul_rn(ri.x, pi.x), ri.y = __dmul_rn(ri.y, pi.y);
      }
      double2 di = d[i];
      di.x = __fma_rn(beta, di.x, ri.x);
      di.y = __fma_rn(beta, di.y, ri.y);
      d[i] = di;
   }
}

// The loop of cg_core splits the updates differently: r first (the stopping test needs it), x together with the
// direction, which reads d anyway: 4 + 6 vector passes per iteration instead of 7 + 4.  Same operations on the same
// operands in the same order as cg_update_xr_kernel + cg_update_dir_kernel, with the roundings pinned by explicit
// __dmul_rn / __fma_rn in all four kernels (left to the compiler, the contraction of B r + beta d differed between the
// two forms): x, r, d are bit-identical (tests/test_gpu_parity.py::test_pcg_matches_building_blocks_bitwise).
// r -= alpha z;  partial <B r, r>
__global__ void __launch_bounds__(kVecThreads)
cg_update_r_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ z,
                   const double2 *__restrict__ dinv, double2 *__restrict__ r, ReduceScratch red, double *__restrict__ out)
{
   if (scal[SC_FLAG] != 0.) return;
   const double alpha = scal[SC_ALPHA];
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n2; i += stride)
   {
      const double2 zi = z[i];
      double2 ri = r[i];
      ri.x = __fma_rn(-alpha, zi.x, ri.x), ri.y = __fma_rn(-alpha, zi.y, ri.y);
      r[i] = ri;
      if (dinv)
      {
         const double2 pi = dinv[i];
         part = __fma_rn(__dmul_rn(pi.x, ri.x), ri.x, part), part = __fma_rn(__dmul_rn(pi.y, ri.y), ri.y, part);
      }
      else
         part = __fma_rn(ri.x, ri.x, part), part = __fma_rn(ri.y, ri.y, part);
   }
   block_reduce_finish<kVecThreads>(part, red, out);
}

// x += alpha d when that update is pending (it is applied even when the iteration stopped: mfem::CGSolver updates x
// before it tests <B r, r>);  then, unless the solve has stopped or x_only, d = B r + beta d
__global__ void __launch_bounds__(kVecThreads)
cg_update_xdir_kernel(int64_t n2, const double *__restrict__ scal, const double2 *__restrict__ r,
                      const double2 *__restrict__ dinv, double2 *__restrict__ x, double2 *__restrict__ d, int x_only)
{
   const bool pend = scal[SC_XPEND] != 0., go = !x_only && scal[SC_FLAG] == 0.;
   if (!pend && !go) return;
   const double alpha = scal[SC_ALPHA], beta = scal[SC_BETA];
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n2; i += stride)
   {
      double2 di = d[i];
      if (pend)
      {
         double2 xi = x[i];
         xi.x = __fma_rn(alpha, di.x, xi.x), xi.y = __fma_rn(alpha, di.y, xi.y);
         x[i] = xi;
      }
      if (go)
      {
         double2 ri = r[i];
         if (dinv)
         {
            const double2 pi = dinv[i];
            ri.x = __dmul_rn(ri.x, pi.x), ri.y = __dmul_rn(ri.y, pi.y);
         }
         di.x = __fma_rn(beta, di.x, ri.x);
         di.y = __fma_rn(beta, di.y, ri.y);
         d[i] = di;
      }
   }
}

__global__ void dinv_kernel(int64_t n, const double *__restrict__ diag, double *__restrict__ dinv)
{
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n) dinv[i] = 1. / diag[i];
}

__global__ void __launch_bounds__(kVecThreads)
dot_kernel(int64_t n, const double *__restrict__ a, const double *__restrict__ b, ReduceScratch red,
           double *__restrict__ out, const double *__restrict__ flag = nullptr)
{
   if (flag && *flag != 0.) return;  // converged CG: keep the previous value
   double part = 0.;
   const int64_t stride = (int64_t)gridDim.x * kVecThreads;
   for (int64_t i = (int64_t)blockIdx.x * kVecThreads + threadIdx.x; i < n; i += stride) part += a[i] * b[i];
   block_reduce_finish<kVecThreads>(part, red, out);
}

// phase 0: after init (nom)   phase 1: after spmv+dot (den)   phase 2: after update_xr (betanom)
// One warp.  With a P2P communicator the all-reduce of the freshly written partial sum is fused in (lane p
// exchanges with rank p, dist.cuh); every rank adds the partials in rank order, so the scalars -- and the
// convergence decisions -- are bit-identical on all ranks.
__global__ void __launch_bounds__(32) cg_scalar_kernel(double *__restrict__ s, int phase, RedArgs ra)
{
   const int idx = phase == 0 ? SC_RED_NOM : (phase == 1 ? SC_RED_DEN : SC_RED_BETA);
   if (ra.hdr)
   {
      double v[1] = {s[idx]};
      __syncwarp();
      mailbox_allreduce<1>(ra, v);
      if (threadIdx.x == 0) s[idx] = v[0];
   }
   if (threadIdx.x != 0) return;
   if (phase == 0)
   {
      const double nom = s[SC_RED_NOM];
      s[SC_NOM] = nom;
      s[SC_R0] = fmax(nom * s[SC_RTOL2], s[SC_ATOL2]);
      s[SC_FINAL] = nom;
      s[SC_ITERS] = 0.;
      // <B r, r> < 0: the preconditioner is not positive definite (mfem::CGSolver::Mult returns unconverged)
      s[SC_FLAG] = (nom < 0.) ? 2. : ((nom <= s[SC_R0]) ? 1. : 0.);
      return;
   }
   if (s[SC_FLAG] != 0.)
   {  // stopped: the direction kernel before this apply has brought x up to date
      if (phase == 1) s[SC_XPEND] = 0.;
      return;
   }
   if (phase == 1)
   {
      const double den = s[SC_RED_DEN];
      s[SC_DEN] = den;
      if (!(den > 0.))
         s[SC_FLAG] = 2., s[SC_XPEND] = 0.;  // not positive definite: mfem leaves the loop before it touches x
      else
         s[SC_ALPHA] = s[SC_NOM] / den, s[SC_XPEND] = 1.;
   }
   else
   {
      const double betanom = s[SC_RED_BETA];
      s[SC_BETANOM] = betanom;
      s[SC_ITERS] += 1.;
      s[SC_FINAL] = betanom;
      if (betanom < 0.)
         s[SC_FLAG] = 2.;
      else if (betanom <= s[SC_R0])
         s[SC_FLAG] = 1.;
      else
      {
         s[SC_BETA] = betanom / s[SC_NOM];
         s[SC_NOM] = betanom;
      }
   }
}

static unsigned vec_grid(int64_t n)
{
   const int64_t want = cdiv(n, kVecThreads);
   const int64_t cap = (int64_t)devinfo().sm_count * 8;  // 8 resident CTAs of 256 threads per SM
   return (unsigned)std::max<int64_t>(1, std::min(want, cap));
}

}  // namespace femb

using namespace femb;

extern "C" int femb200_dot(int64_t n, const double *d_a, const double *d_b, double *d_out, void *stream)
{
   FEMB_CHECK(d_a && d_b && d_out && n >= 0, "dot: bad argument");
   cudaStream_t st = as_stream(stream);
   const unsigned grid = vec_grid(n);
   ReduceScratch red;
   if (int rc = reduce_scratch(grid, st, &red)) return rc;
   dot_kernel<<<grid, kVecThreads, 0, st>>>(n, d_a, d_b, red, d_out);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_jacobi_setup(int64_t n, const double *d_diag, double *d_dinv, void *stream)
{
   FEMB_CHECK(d_diag && d_dinv && n >= 0, "jacobi_setup: bad argument");
   dinv_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(n, d_diag, d_dinv);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_cg_set_tolerances(double *d_scal, double rtol, double atol, void *stream)
{
   FEMB_CHECK(d_scal, "cg_set_tolerances: null scalars");
   double h[SC_COUNT];
   for (int i = 0; i < SC_COUNT; ++i) h[i] = 0.;
   h[SC_RTOL2] = rtol * rtol;
   h[SC_ATOL2] = atol * atol;
   // pageable source: the copy is staged before the call returns
   FEMB_CUDA(cudaMemcpyAsync(d_scal, h, sizeof(h), cudaMemcpyHostToDevice, as_stream(stream)));
   return 0;
}

extern "C" int femb200_cg_init(int64_t n, const double *d_b, const double *d_dinv, double *d_x, double *d_r,
                               double *d_dir, double *d_scal, void *stream)
{
   FEMB_CHECK(d_b && d_x && d_r && d_dir && d_scal && n >= 0, "cg_init: bad argument");
   cudaStream_t st = as_stream(stream);
   const unsigned grid = vec_grid(n);
   ReduceScratch red;
   if (int rc = reduce_scratch(grid, st, &red)) return rc;
   cg_init_kernel<<<grid, kVecThreads, 0, st>>>(n, d_b, d_dinv, d_x, d_r, d_dir, red, d_scal + SC_RED_NOM);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_cg_scalar_step(double *d_scal, int phase, void *stream)
{
   FEMB_CHECK(d_scal && phase >= 0 && phase <= 2, "cg_scalar_step: bad argument");
   cg_scalar_kernel<<<1, 32, 0, as_stream(stream)>>>(d_scal, phase, RedArgs());
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_cg_update_xr(int64_t n, double *d_scal, const double *d_dir, const double *d_Ad,
                                    const double *d_dinv, double *d_x, double *d_r, void *stream)
{
   FEMB_CHECK(d_scal && d_dir && d_Ad && d_x && d_r && n >= 0 && (n & 1) == 0, "cg_update_xr: bad argument");
   cudaStream_t st = as_stream(stream);
   const unsigned grid = vec_grid(n / 2);
   ReduceScratch red;
   if (int rc = reduce_scratch(grid, st, &red)) return rc;
   cg_update_xr_kernel<<<grid, kVecThreads, 0, st>>>(
       n / 2, d_scal, reinterpret_cast<const double2 *>(d_dir), reinterpret_cast<const double2 *>(d_Ad),
       reinterpret_cast<const double2 *>(d_dinv), reinterpret_cast<double2 *>(d_x), reinterpret_cast<double2 *>(d_r),
       red, d_scal + SC_RED_BETA);
   FEMB_LAUNCH_CHECK();
   return 0;
}

extern "C" int femb200_cg_update_dir(int64_t n, const double *d_scal, const double *d_r, const double *d_dinv,
                                     double *d_dir, void *stream)
{
   FEMB_CHECK(d_scal && d_r && d_dir && n >= 0 && (n & 1) == 0, "cg_update_dir: bad argument");
   cg_update_dir_kernel<<<vec_grid(n / 2), kVecThreads, 0, as_stream(stream)>>>(
       n / 2, d_scal, reinterpret_cast<const double2 *>(d_r), reinterpret_cast<const double2 *>(d_dinv),
       reinterpret_cast<double2 *>(d_dir));
   FEMB_LAUNCH_CHECK();
   return 0;
}

namespace femb {

// z = A d on the owned rows with the fused partial <d, A d> into scal[SC_RED_DEN]; no-op once the flag is set
// The matrix-free operator of a rank works on its whole local mesh (owned + ghost cells): the rows of the owned
// nodes are complete, those of ghost nodes are partial and ignored, so with a partition the fused <d, A d> of the
// apply kernel (a sum over every local node) is replaced by a dot product over the owned dofs.
// compact: the mode of spmv_launch (0 on the matrix-free operator)
static int cg_apply_rows(const femb200_plan *plan, int op_kind, const void *op, const double *d_values, const RowRange &rr,
                         int64_t own_lo, int64_t own_hi, const double *d_dir, double *d_Ad, double *d_scal, cudaStream_t st,
                         int compact = 0)
{
   if (op_kind == FEMB200_OP_CSR)
      return spmv_launch(plan, rr, d_values, d_dir, d_Ad, d_scal + SC_FLAG, d_scal + SC_RED_DEN, false, st, compact);
   const femb200_pa *pa = static_cast<const femb200_pa *>(op);
   if (own_lo == 0 && 2 * own_hi == pa_num_dofs(pa))
      return pa_apply_launch(pa, d_dir, d_Ad, d_scal + SC_FLAG, d_scal + SC_RED_DEN, st, false);
   if (int rc = pa_apply_launch(pa, d_dir, d_Ad, d_scal + SC_FLAG, nullptr, st, false)) return rc;
   const int64_t n = 2 * (own_hi - own_lo);
   const unsigned grid = vec_grid(n);
   ReduceScratch red;
   if (int rc = reduce_scratch(grid, st, &red)) return rc;
   dot_kernel<<<grid, kVecThreads, 0, st>>>(n, d_dir + 2 * own_lo, d_Ad + 2 * own_lo, red, d_scal + SC_RED_DEN, d_scal + SC_FLAG);
   FEMB_LAUNCH_CHECK();
   return 0;
}

// The PCG loop of femb200_pcg and femb200_dist_pcg.  Vector kernels run on the owned dofs [2 own_lo,
// 2 own_hi) of the local vectors; with a communicator the search direction gets its ghost update before
// every operator apply and the three dot products are all-reduced (fused into the scalar kernels on the P2P
// transport, ncclAllReduce on the NCCL transport).  With use_graph the full iteration (update_r, scalar,
// update_xdir, ghost update, apply + dot, scalar) is captured once into a CUDA graph cached in the
// communicator and replayed; everything it needs (scalars, sequence numbers) lives in device memory.
// On a plan with compact values (plan.cuh) the first apply also writes the kept blocks of this solve's values into the
// plan's compact copy and checks the dropped ones; the applies of the loop then stream the copy (about a quarter fewer
// bytes on P2), or the CSR values when a dropped block was not zero.  Both give the same bits.  The copy belongs to
// the plan: solves on one plan must not run concurrently.
int cg_core(const CgProblem &P, int *iters, double *final_norm, int *converged, cudaStream_t st)
{
   const int64_t o = 2 * P.own_lo, n = 2 * (P.own_hi - P.own_lo);
   const double *dinv_o = P.dinv ? P.dinv + o : nullptr;
   double *scal = P.scal;
   RowRange rr{0, 0, {0, 0}, 0};
   int compact = 0;
   if (P.op_kind == FEMB200_OP_CSR)
   {
      FEMB_CHECK(P.plan && P.values, "pcg: the CSR operator needs a plan and values");
      if (int rc = plan_row_range(P.plan, P.own_lo, P.own_hi, &rr)) return rc;
      femb200_plan *pm = const_cast<femb200_plan *>(P.plan);
      compact = spmv_compact_ready(pm, rr) ? 2 : 0;
   }
   else
      FEMB_CHECK(P.op_kind == FEMB200_OP_PA && P.op, "pcg: unknown operator kind %d", P.op_kind);
   const RedArgs ra = dist_red_args(P.comm);
   const unsigned gv = vec_grid(n / 2), gi = vec_grid(n);
   ReduceScratch red;
   if (int rc = reduce_scratch(std::max(gv, gi), st, &red)) return rc;  // grown before any capture
   int rc;
   auto scalar = [&](int phase, int idx, cudaStream_t s) -> int {
      if (int e = dist_allreduce_pre(P.comm, scal + idx, 1, s)) return e;
      cg_scalar_kernel<<<1, 32, 0, s>>>(scal, phase, ra);
      FEMB_LAUNCH_CHECK();
      return 0;
   };
   auto apply = [&](cudaStream_t s, int cmode) -> int {
      if (int e = dist_halo_arena(P.comm, s)) return e;
      if (int e = cg_apply_rows(P.plan, P.op_kind, P.op, P.values, rr, P.own_lo, P.own_hi, P.d, P.z, scal, s, cmode)) return e;
      return scalar(1, SC_RED_DEN, s);
   };
   auto update_r = [&](cudaStream_t s) -> int {
      ReduceScratch rs;
      if (int e = reduce_scratch(gv, s, &rs)) return e;
      cg_update_r_kernel<<<gv, kVecThreads, 0, s>>>(n / 2, scal, reinterpret_cast<const double2 *>(P.z + o),
                                                    reinterpret_cast<const double2 *>(dinv_o), reinterpret_cast<double2 *>(P.r + o),
                                                    rs, scal + SC_RED_BETA);
      FEMB_LAUNCH_CHECK();
      return scalar(2, SC_RED_BETA, s);
   };
   auto update_xdir = [&](cudaStream_t s, int x_only) -> int {
      cg_update_xdir_kernel<<<gv, kVecThreads, 0, s>>>(n / 2, scal, reinterpret_cast<const double2 *>(P.r + o),
                                                       reinterpret_cast<const double2 *>(dinv_o), reinterpret_cast<double2 *>(P.x + o),
                                                       reinterpret_cast<double2 *>(P.d + o), x_only);
      FEMB_LAUNCH_CHECK();
      return 0;
   };
   auto full_iteration = [&](cudaStream_t s) -> int {
      if (int e = update_r(s)) return e;
      if (int e = update_xdir(s, 0)) return e;
      return apply(s, compact);
   };

   if ((rc = femb200_cg_set_tolerances(scal, P.rtol, P.atol, st))) return rc;
   cg_init_kernel<<<gi, kVecThreads, 0, st>>>(n, P.b + o, dinv_o, P.x + o, P.r + o, P.d + o, red, scal + SC_RED_NOM);
   FEMB_LAUNCH_CHECK();
   if ((rc = scalar(0, SC_RED_NOM, st))) return rc;
   if (compact) FEMB_CUDA(cudaMemsetAsync(P.plan->cbad, 0, sizeof(int), st));
   if ((rc = apply(st, compact ? 1 : 0))) return rc;

   const int nit = P.fixed_iters > 0 ? P.fixed_iters : P.maxit;
   const int check_every = P.check_every > 0 ? P.check_every : 25;
   double hs[SC_COUNT];
   bool stopped = false;
   // iterations 1 .. nit - 1 are full ones; the last one stops after the residual update
   IterGraph *G = (P.use_graph && P.comm && nit >= 4) ? dist_iter_graph(P.comm) : nullptr;
   for (int i = 1; i <= nit && !stopped; ++i)
   {
      if (i == nit)
      {
         if ((rc = update_r(st))) return rc;
         if ((rc = update_xdir(st, 1))) return rc;
      }
      else if (G && i >= 2)
      {  // iteration 1 ran eagerly (warm kernels, NCCL connections); capture on first use, then replay
         const void *key[8] = {P.plan, P.op, P.values, P.x, P.r, P.d, P.z, P.dinv};
         const int64_t ikey[4] = {P.own_lo, P.own_hi, (int64_t)P.op_kind, (int64_t)compact};
         if (!G->exec || memcmp(G->key, key, sizeof(key)) || memcmp(G->ikey, ikey, sizeof(ikey)))
         {
            if (G->exec) cudaGraphExecDestroy(G->exec), G->exec = nullptr;
            // captured on the communicator's own stream (the caller's may be the legacy default stream, which
            // cannot be captured); the fused-reduction scratch of that stream is created before the capture
            cudaStream_t cs = dist_capture_stream(P.comm);
            FEMB_CHECK(cs != nullptr, "pcg: no capture stream");
            ReduceScratch warm;
            if (int e = reduce_scratch(4096, cs, &warm)) return e;
            FEMB_CUDA(cudaStreamSynchronize(cs));
            cudaGraph_t graph = nullptr;
            FEMB_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            const int e = full_iteration(cs);
            const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
            if (e || ce != cudaSuccess || !graph)
            {
               if (graph) cudaGraphDestroy(graph);
               if (e) return e;
               return set_error("pcg: capturing the iteration graph failed: %s", cudaGetErrorString(ce));
            }
            const cudaError_t ie = cudaGraphInstantiate(&G->exec, graph, 0);
            cudaGraphDestroy(graph);
            FEMB_CHECK(ie == cudaSuccess, "pcg: cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
            memcpy(G->key, key, sizeof(key)), memcpy(G->ikey, ikey, sizeof(ikey));
         }
         FEMB_CUDA(cudaGraphLaunch(G->exec, st));
      }
      else if ((rc = full_iteration(st)))
         return rc;
      if (P.fixed_iters <= 0 && (i % check_every == 0) && i < nit)
      {
         FEMB_CUDA(cudaMemcpyAsync(hs, scal, sizeof(hs), cudaMemcpyDeviceToHost, st));
         FEMB_CUDA(cudaStreamSynchronize(st));
         stopped = hs[SC_FLAG] != 0.;
      }
   }
   FEMB_CUDA(cudaMemcpyAsync(hs, scal, sizeof(hs), cudaMemcpyDeviceToHost, st));
   FEMB_CUDA(cudaStreamSynchronize(st));
   if ((rc = dist_check_error(P.comm, st))) return rc;
   const bool conv = hs[SC_FLAG] == 1.;
   if (converged) *converged = conv ? 1 : 0;
   // mfem::CGSolver: final_iter = the iteration it stopped in (convergence or breakdown), max_iter otherwise
   if (iters) *iters = (conv || hs[SC_FLAG] == 2. || P.fixed_iters > 0) ? (int)hs[SC_ITERS] : P.maxit;
   if (final_norm) *final_norm = sqrt(hs[SC_FINAL] > 0. ? hs[SC_FINAL] : 0.);
   return 0;
}

}  // namespace femb

// z = A d with the fused partial <d, A d> into scal[SC_RED_DEN]; no-op once the flag is set
extern "C" int femb200_cg_apply(const femb200_plan *plan, int op_kind, const void *op, const double *d_values,
                                const double *d_dir, double *d_Ad, double *d_scal, void *stream)
{
   FEMB_CHECK(d_dir && d_Ad && d_scal, "cg_apply: null argument");
   RowRange rr{0, 0, {0, 0}, 0};
   if (op_kind == FEMB200_OP_CSR)
   {
      FEMB_CHECK(plan && d_values, "cg_apply: CSR operator needs a plan and values");
      if (int rc = plan_row_range(plan, 0, plan->nnodes, &rr)) return rc;
   }
   else
      FEMB_CHECK(op_kind == FEMB200_OP_PA && op, "cg_apply: unknown operator kind %d", op_kind);
   return cg_apply_rows(plan, op_kind, op, d_values, rr, 0, op_kind == FEMB200_OP_CSR ? plan->nnodes : pa_num_dofs(static_cast<const femb200_pa *>(op)) / 2,
                        d_dir, d_Ad, d_scal, as_stream(stream));
}

extern "C" int femb200_pcg(const femb200_plan *plan, int op_kind, const void *op, const double *d_values,
                           const double *d_b, double *d_x, int64_t n, double rtol, double atol, int maxit,
                           const double *d_dinv, int check_every, int fixed_iters, double *d_work, int *iters,
                           double *final_norm, int *converged, void *stream)
{
   FEMB_CHECK(d_b && d_x && d_work && n > 0 && (n & 1) == 0, "pcg: bad argument");
   FEMB_CHECK(maxit >= 0, "pcg: negative maxit");
   if (op_kind == FEMB200_OP_CSR)
      FEMB_CHECK(plan && n == 2 * plan->nnodes, "pcg: n = %lld does not match the operator (%lld dofs)", (long long)n,
                 (long long)(plan ? 2 * plan->nnodes : 0));
   else if (op_kind == FEMB200_OP_PA && op)
      FEMB_CHECK(n == pa_num_dofs(static_cast<const femb200_pa *>(op)), "pcg: n = %lld does not match the matrix-free operator",
                 (long long)n);
   CgProblem P;
   P.plan = plan, P.op_kind = op_kind, P.op = op, P.values = d_values;
   P.own_lo = 0, P.own_hi = n / 2;
   P.b = d_b, P.dinv = d_dinv, P.x = d_x;
   P.r = d_work, P.d = d_work + n, P.z = d_work + 2 * n, P.scal = d_work + 3 * n;
   P.rtol = rtol, P.atol = atol, P.maxit = maxit, P.check_every = check_every, P.fixed_iters = fixed_iters;
   return cg_core(P, iters, final_norm, converged, as_stream(stream));
}

// dst[k] = src[idx[k]] over node pairs (16-byte items): packs the interface dofs
// of a halo message (role of the dolfinx Scatterer pack step behind
// VecGhostUpdate(INSERT, FORWARD), F.cc:865-866)
namespace femb {
__global__ void gather_kernel(int64_t n, const int32_t *__restrict__ idx, const double2 *__restrict__ src,
                              double2 *__restrict__ dst)
{
   const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (k < n) dst[k] = src[idx[k]];
}
}  // namespace femb

extern "C" int femb200_gather(int64_t nnodes_out, const int32_t *d_node_idx, const double *d_src, double *d_dst,
                              void *stream)
{
   FEMB_CHECK(nnodes_out >= 0 && (nnodes_out == 0 || (d_node_idx && d_src && d_dst)), "gather: bad argument");
   if (nnodes_out == 0) return 0;
   femb::gather_kernel<<<(unsigned)cdiv(nnodes_out, 256), 256, 0, as_stream(stream)>>>(
       nnodes_out, d_node_idx, reinterpret_cast<const double2 *>(d_src), reinterpret_cast<double2 *>(d_dst));
   FEMB_LAUNCH_CHECK();
   return 0;
}

// dst[idx[k]] = src[k] over nodes of `width` doubles (2 or 3): uploads the coordinates of the
// geometry vertices only (dolfinx keeps the P1 geometry apart from the P2 space: mesh.geometry.x
// holds the vertices, F.cc:213), the edge nodes of a straight-sided P2 mesh are never read
namespace femb {
__global__ void scatter_rows_kernel(int64_t n, int width, const int32_t *__restrict__ idx, const double *__restrict__ src,
                                    double *__restrict__ dst)
{
   const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (k >= n) return;
   const int64_t j = idx[k];
   for (int c = 0; c < width; ++c) dst[j * width + c] = src[k * width + c];
}
}  // namespace femb

extern "C" int femb200_scatter_rows(int64_t n, int width, const int32_t *d_idx, const double *d_src, double *d_dst,
                                    void *stream)
{
   FEMB_CHECK(n >= 0 && width >= 1 && width <= 3 && (n == 0 || (d_idx && d_src && d_dst)), "scatter_rows: bad argument");
   if (n == 0) return 0;
   femb::scatter_rows_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(n, width, d_idx, d_src, d_dst);
   FEMB_LAUNCH_CHECK();
   return 0;
}
