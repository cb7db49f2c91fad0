// topolow_b200/csrc/tiledev.h - device-side views shared by every instantiation of the tile kernel.
#pragma once
#include "schedule.h"

namespace tl {

// Coordinates given to phantom (padding) slots: far away in FP32 so that their force underflows to
// zero (tilepass.cuh, FastF32), zero in the exact policy (which tests the mass instead).
constexpr float kPhantomCoordF32 = 1.0e18f;
constexpr double kPhantomCoordF64 = 0.0;

struct __align__(16) EdgeRec {
  double target;
  uint32_t slot_lo;        // slot in the lower-numbered tile (or lower slot when same tile)
  uint32_t slot_hi_type;   // slot in the other tile | type << 30   (0 exact, 1 '>', 2 '<')
};

template <class real>
struct TileDev {
  real* pos;
  real* best;
  const real* dp1;
  const EdgeRec* edges;
  const uint32_t* bucket_off;
  FitState* state;
  double* partials;      // [G][4]: error sum, count, non-finite flag, unused
  unsigned* barrier;     // [0] arrivals, [1] generation of the grid barrier; [32 + b]: round counter of super-block b
  double* trace;         // [n_iter] or null
  long long n_edges;
  unsigned long long pairs_per_iter;
  const volatile int* abort;   // mapped host word: non-zero = the caller asks the fit to stop (null = never)
};

// One entry of a many-fits launch (tile_batch_kernel).
template <class real>
struct BatchJob {
  TileDev<real> dv;
  Geometry geo;
  FitParams prm;
  int n_iters;
  int pad;
  volatile int* host_flag;
};

}  // namespace tl
