// cg_slots.cuh -- slots of the 16 device-resident CG scalars (femb200.h, "CG building blocks"), shared by the
// Jacobi PCG (cg.cu) and the multigrid PCG (mg.cu), which drive the same scalar kernel.
#pragma once
#include "../../include/femb200.h"

namespace femb {

enum
{
   SC_NOM = 0,
   SC_DEN = 1,
   SC_BETANOM = 2,
   SC_R0 = 3,
   SC_FLAG = 4,
   SC_ITERS = 5,
   SC_FINAL = 6,
   SC_RTOL2 = 7,
   SC_ATOL2 = 8,
   SC_RED_NOM = 9,   // local (per-rank) sums written by the vector kernels
   SC_RED_DEN = 10,
   SC_RED_BETA = 11,
   SC_BETA = 12,
   SC_ALPHA = 13,  // nom / den of the current iteration (cg_core: the x update is deferred to the direction kernel)
   SC_XPEND = 14,  // 1 while x += alpha d of the current iteration has not been applied yet
   SC_COUNT = 16
};

static_assert(SC_FLAG == FEMB200_SC_FLAG && SC_ITERS == FEMB200_SC_ITERS && SC_FINAL == FEMB200_SC_FINAL &&
                  SC_RED_NOM == FEMB200_SC_RED_NOM && SC_RED_DEN == FEMB200_SC_RED_DEN &&
                  SC_RED_BETA == FEMB200_SC_RED_BETA && SC_COUNT == FEMB200_SC_COUNT,
              "CG scalar slots disagree with femb200.h");

}  // namespace femb
