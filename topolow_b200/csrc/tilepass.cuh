// topolow_b200/csrc/tilepass.cuh
//
// PRODUCTION KERNEL (TOPOLOW_MODE_COLOURED): one persistent kernel runs whole iterations of
// the reference's pair loop (src/optimization.cpp:193-366) - all N(N-1)/2 pair updates, the
// cooling step (:289), the edge MAE (:54-81, :294-296), the three-way convergence controller
// with best-state snapshot (:303-357) and the finite check (:359-361) - with no host
// round-trip.  The pair order is the structured permutation defined in schedule.h.
//
// Data layout in HBM
//   pos / best : [slot][D] reals (AoS; slot = position of a point after the initial random
//                relabelling, 64 consecutive slots = one tile, padded with phantom slots)
//   dp1        : [slot] (degree + 1), 0 marks a phantom slot
//   edges      : 16-byte records {double target; u32 slot_lo; u32 slot_hi | type << 30},
//                counting-sorted by (tile_lo, tile_hi); bucket_off[tile_lo * T + tile_hi]
// On chip
//   the 2W tiles of a CTA task sit in shared memory as [k][65] (dimension-major, padded);
//   during a tile x tile pass lane a holds kP A points (slots a, a+32, ..) and kP travelling B
//   points in registers - kP*kP pair updates per ring step, kP of them independent at a time -
//   and the B points move with warp shuffles; measured pairs of the tile pair are scattered
//   into a per-warp kP*kP x 32 x 32 target table + 2*kP*kP 32-bit lane masks before the pass.
#pragma once

#include "tiledev.h"

#ifndef TL_KP
#error "define TL_KP (points per lane: 1, 2 or 3) before including tilepass.cuh"
#endif
#ifndef TL_RING_UNROLL
#define TL_RING_UNROLL 0   // ring steps per loop trip; 0 = the measured default per tile size (kRingUnroll)
#endif
#define TL_PNS_CAT2(a, b) a##b
#define TL_PNS_CAT(a, b) TL_PNS_CAT2(a, b)
#define TL_PNS TL_PNS_CAT(p, TL_KP)

namespace tl {
namespace TL_PNS {   // one copy of everything below per tile size

constexpr int kP = TL_KP;        // points of a tile held by one lane
constexpr int kTile = 32 * kP;   // points per tile
// Ring steps per loop trip.  Inside an unrolled trip the shuffles of a step are scheduled between the
// FMAs of the next one; only the last step of a trip has nothing after it.  Measured on B200 (ms per
// iteration at N = 100k, d = 16, 96-point tiles): 1 -> 25.3, 2 -> 23.7, 4 -> 22.7, 8 -> 22.7; the smaller
// bodies of the 32- and 64-point kernels gain a little more from 8.
constexpr int kRingUnroll = TL_RING_UNROLL ? TL_RING_UNROLL : (kP == 3 ? 4 : 8);

// ---------------------------------------------------------------------------------------
// Math policies.  A policy owns the register image of a point (`Point<D>`: coordinates + the
// mass terms that travel with it) and the arithmetic of one pair visit.
// ---------------------------------------------------------------------------------------

// One pair visit's measurement.  `pos` / `neg` are zero or non-zero words (the lane's masks ANDed with
// the step bit): pos = the pair pulls when the embedded distance is BELOW the target (an exact value
// or a '>' threshold, src/optimization.cpp:237-239), neg = it pulls when ABOVE (exact or '<', :240-242).
// Both zero = unmeasured pair; `target` is only meaningful otherwise.
template <class real>
struct Cell {
  real target;
  uint32_t pos, neg;
};

constexpr int kRow = kTile + 1;   // shared-memory row of one dimension: kTile slots + 1 pad (kTile % 32 == 0)

// Two FP32 values in one 64-bit register: sm_100 has 2-wide FP32 FMA/ADD/MUL (SASS FFMA2 ...),
// which halves the instruction count of the coordinate loops.
typedef float2 f32x2;
TL_D f32x2 pk2(float lo, float hi) { return make_float2(lo, hi); }
TL_D void upk2(f32x2 v, float& lo, float& hi) { lo = v.x; hi = v.y; }
TL_D f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { return __ffma2_rn(a, b, c); }
TL_D f32x2 mul2(f32x2 a, f32x2 b) { return __fmul2_rn(a, b); }
TL_D f32x2 add2(f32x2 a, f32x2 b) { return __fadd2_rn(a, b); }
TL_D float sqrt_fast(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
TL_D float rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// FP32 production arithmetic.  A phantom slot (padding of the last tile) has zero mass and sits
// at kPhantomCoordF32 in every dimension: against a real point 1/ds^3 flushes to zero, against
// another phantom the zero mass cancels the force, so no validity predicate is needed.
struct FastF32 {
  typedef float real;
  static constexpr int kMaxWarps = kP == 1 ? 16 : (kP == 2 ? 8 : 4);   // shared memory (kP*kP target tables per warp), registers
  struct Ctx { float two_k, c_half, k; };
  static TL_D Ctx make_ctx(double k, double c_rep) {
    Ctx c; c.two_k = (float)(2.0 * k); c.c_half = (float)(0.5 * c_rep); c.k = (float)k; return c;
  }
  template <int D>
  struct Point {
    static constexpr int H = (D + 1) / 2;
    f32x2 c[H];       // coordinates, two per register (odd D: the last high half is 0)
    float rdeg;       // (c / 2) / (deg + 1)      repulsion weight, constant folded in (0 for a phantom)
    float rnorm;      // 2k / (4 (deg + 1) + k)   spring weight, constant folded in    (0 for a phantom)
    TL_D void load(const float* s, int idx, const Ctx& ctx) {
#pragma unroll
      for (int j = 0; j < H; ++j)
        c[j] = pk2(s[(2 * j) * kRow + idx], (2 * j + 1 < D) ? s[(2 * j + 1) * kRow + idx] : 0.f);
      const float dp1 = s[D * kRow + idx];
      const bool ok = dp1 > 0.f;
      rdeg = ok ? ctx.c_half * rcp_fast(dp1) : 0.f;
      rnorm = ok ? ctx.two_k * rcp_fast(fmaf(4.0f, dp1, ctx.k)) : 0.f;
    }
    TL_D void store(float* s, int idx) const {
#pragma unroll
      for (int j = 0; j < H; ++j) {
        float lo, hi;
        upk2(c[j], lo, hi);
        s[(2 * j) * kRow + idx] = lo;
        if (2 * j + 1 < D) s[(2 * j + 1) * kRow + idx] = hi;
      }
    }
    TL_D void shfl_from(int src) {
      const unsigned full = 0xffffffffu;
#pragma unroll
      for (int j = 0; j < H; ++j) {
        float lo, hi;
        upk2(c[j], lo, hi);
        lo = __shfl_sync(full, lo, src);
        if (2 * j + 1 < D) hi = __shfl_sync(full, hi, src);
        c[j] = pk2(lo, hi);
      }
      rdeg = __shfl_sync(full, rdeg, src);
      rnorm = __shfl_sync(full, rnorm, src);
    }
    TL_D void shfl_xor_of(const Point& o, int x) {
      const unsigned full = 0xffffffffu;
#pragma unroll
      for (int j = 0; j < H; ++j) {
        float lo, hi;
        upk2(o.c[j], lo, hi);
        lo = __shfl_xor_sync(full, lo, x);
        if (2 * j + 1 < D) hi = __shfl_xor_sync(full, hi, x);
        c[j] = pk2(lo, hi);
      }
      rdeg = __shfl_xor_sync(full, o.rdeg, x);
      rnorm = __shfl_xor_sync(full, o.rnorm, x);
    }
  };

  // delta = B - A, and the scalar with which it is applied to each endpoint
  // (src/optimization.cpp:207-281 with reciprocals hoisted out of the coordinate loop).
  static TL_D bool is_spring(float target_minus_dist, const Cell<float>& cell) {
    return (target_minus_dist > 0.f ? cell.pos : cell.neg) != 0u;
  }
  template <int D>
  static TL_D void force(const Point<D>& A, const Point<D>& B, f32x2 (&delta)[Point<D>::H], const Cell<float>& cell,
                         const Ctx& c, float& fA, float& fB) {
    constexpr int H = Point<D>::H;
    const float target = cell.target;
    const f32x2 neg1 = pk2(-1.0f, -1.0f);
#pragma unroll
    for (int j = 0; j < H; ++j) delta[j] = fma2(A.c[j], neg1, B.c[j]);
    f32x2 acc0 = mul2(delta[0], delta[0]);
    f32x2 acc1 = pk2(0.f, 0.f);
    if (H > 1) acc1 = mul2(delta[1], delta[1]);
#pragma unroll
    for (int j = 2; j < H; ++j) {
      if (j & 1) acc1 = fma2(delta[j], delta[j], acc1);
      else acc0 = fma2(delta[j], delta[j], acc0);
    }
    if (H > 1) acc0 = add2(acc0, acc1);
    float lo, hi;
    upk2(acc0, lo, hi);
    const float dist = sqrt_fast(lo + hi);
    const float ids = rcp_fast(dist + 0.01f);
    // Branch-free choice between repulsion c / (2 ds^3) and spring 2k (t - d) / ds: the target cell is
    // read unconditionally (stale / garbage when the pair is not measured; then both masks are zero
    // and the selects discard it).  One compare picks the mask that applies on this side of the target.
    // (At dist == target exactly a '<' pair gets the zero spring force instead of the repulsion.)
    const float spr = target - dist;
    const bool spring = is_spring(spr, cell);
    const float rep = ids * ids;            // (c/2 and 2k live in the per-point weights)
    const float f = (spring ? spr : rep) * ids;
    const float wA = spring ? A.rnorm : A.rdeg, wB = spring ? B.rnorm : B.rdeg;
    fA = f * wA;
    fB = f * wB;
  }
  template <int D>
  static TL_D void pair(Point<D>& A, Point<D>& B, const Cell<float>& cell, const Ctx& c) {
    constexpr int H = Point<D>::H;
    f32x2 delta[H];
    float fA, fB;
    force<D>(A, B, delta, cell, c, fA, fB);
    const f32x2 nA = pk2(-fA, -fA), pB = pk2(fB, fB);
#pragma unroll
    for (int j = 0; j < H; ++j) {
      A.c[j] = fma2(delta[j], nA, A.c[j]);
      B.c[j] = fma2(delta[j], pB, B.c[j]);
    }
  }
  // One wave: kP independent pair visits (A[p], B[q(p)]) written in lock-step so that their dependency
  // chains (distance -> rsqrt -> rcp -> factors) overlap.  q(p) = (p + w) % kP (kSum = false, ring pass)
  // or (w - p) mod kP (kSum = true, intra pass: symmetric under swapping the two lanes).
  // kRotate (last wave of a ring step): every B point moves on to lane `src` as soon as its update is
  // written, so that the shuffles issue between the FMAs of the A updates instead of after them.
  template <int D, int W_, bool kSum, bool kRotate>
  static TL_D void wave(Point<D> (&A)[kP], Point<D> (&B)[kP], const Cell<float> (&cell)[kP], const Ctx& c, int src) {
    constexpr int H = Point<D>::H;
    const f32x2 neg1 = pk2(-1.0f, -1.0f);
    f32x2 d[kP][H];
    float f[kP];
    bool sp[kP];
#pragma unroll
    for (int j = 0; j < H; ++j)
#pragma unroll
      for (int p = 0; p < kP; ++p) {
        const int q = kSum ? (W_ - p + kP) % kP : (p + W_) % kP;
        d[p][j] = fma2(A[p].c[j], neg1, B[q].c[j]);
      }
    // squared distance: one accumulator chain per visit when kP visits interleave (their chains hide
    // each other's latency and every instruction counts), two when the lane has a single visit
    constexpr int kAcc = (kP == 1 && H > 1) ? 2 : 1;
    f32x2 acc[kP][kAcc];
#pragma unroll
    for (int j = 0; j < H; ++j)
#pragma unroll
      for (int p = 0; p < kP; ++p)
        acc[p][j % kAcc] = j < kAcc ? mul2(d[p][j], d[p][j]) : fma2(d[p][j], d[p][j], acc[p][j % kAcc]);
    float dist[kP], ids[kP];
#pragma unroll
    for (int p = 0; p < kP; ++p) {
      const f32x2 t = kAcc > 1 ? add2(acc[p][0], acc[p][kAcc - 1]) : acc[p][0];
      dist[p] = sqrt_fast(t.x + t.y);
    }
#pragma unroll
    for (int p = 0; p < kP; ++p) ids[p] = rcp_fast(dist[p] + 0.01f);
#pragma unroll
    for (int p = 0; p < kP; ++p) {
      const float spr = cell[p].target - dist[p];
      sp[p] = is_spring(spr, cell[p]);
      f[p] = (sp[p] ? spr : ids[p] * ids[p]) * ids[p];   // x weight: 2k(t-d)/ds or c/(2 ds^3)
    }
    if (!kRotate) {
#pragma unroll
      for (int p = 0; p < kP; ++p) {
        const int q = kSum ? (W_ - p + kP) % kP : (p + W_) % kP;
        const float fA = f[p] * (sp[p] ? A[p].rnorm : A[p].rdeg), fB = f[p] * (sp[p] ? B[q].rnorm : B[q].rdeg);
        const f32x2 nA = pk2(-fA, -fA), pB = pk2(fB, fB);
#pragma unroll
        for (int j = 0; j < H; ++j) {
          A[p].c[j] = fma2(d[p][j], nA, A[p].c[j]);
          B[q].c[j] = fma2(d[p][j], pB, B[q].c[j]);
        }
      }
    } else {
      float fA[kP];
#pragma unroll
      for (int p = 0; p < kP; ++p) {
        const int q = kSum ? (W_ - p + kP) % kP : (p + W_) % kP;
        fA[p] = f[p] * (sp[p] ? A[p].rnorm : A[p].rdeg);
        const float fB = f[p] * (sp[p] ? B[q].rnorm : B[q].rdeg);
        const f32x2 pB = pk2(fB, fB);
#pragma unroll
        for (int j = 0; j < H; ++j) B[q].c[j] = fma2(d[p][j], pB, B[q].c[j]);
      }
#pragma unroll
      for (int q = 0; q < kP; ++q) B[q].shfl_from(src);
#pragma unroll
      for (int p = 0; p < kP; ++p) {
        const f32x2 nA = pk2(-fA[p], -fA[p]);
#pragma unroll
        for (int j = 0; j < H; ++j) A[p].c[j] = fma2(d[p][j], nA, A[p].c[j]);
      }
    }
  }
};

// IEEE double, one rounding per reference operation, no FMA contraction: bit-comparable with
// the CPU loop executed on the order topolow_plan_enumerate() reports.
struct ExactF64 {
  typedef double real;
  static constexpr int kMaxWarps = kP == 1 ? 8 : (kP == 2 ? 4 : 2);  // shared memory: kP*kP x 32 x 32 doubles of targets per warp
  struct Ctx { double k, c_rep; };
  static TL_D Ctx make_ctx(double k, double c_rep) { Ctx c; c.k = k; c.c_rep = c_rep; return c; }
  template <int D>
  struct Point {
    double c[D];
    double dp1;   // deg + 1, 0 = phantom
    TL_D void load(const double* s, int idx, const Ctx&) {
#pragma unroll
      for (int k = 0; k < D; ++k) c[k] = s[k * kRow + idx];
      dp1 = s[D * kRow + idx];
    }
    TL_D void store(double* s, int idx) const {
#pragma unroll
      for (int k = 0; k < D; ++k) s[k * kRow + idx] = c[k];
    }
    TL_D void shfl_from(int src) {
#pragma unroll
      for (int k = 0; k < D; ++k) c[k] = __shfl_sync(0xffffffffu, c[k], src);
      dp1 = __shfl_sync(0xffffffffu, dp1, src);
    }
    TL_D void shfl_xor_of(const Point& o, int x) {
#pragma unroll
      for (int k = 0; k < D; ++k) c[k] = __shfl_xor_sync(0xffffffffu, o.c[k], x);
      dp1 = __shfl_xor_sync(0xffffffffu, o.dp1, x);
    }
  };
  template <int D>
  static TL_D void scalars(const double (&delta)[D], const Cell<double>& cell, const Ctx& c, bool& spring,
                           double& factor) {
    double dist_sq = 0.0;
#pragma unroll
    for (int k = 0; k < D; ++k) dist_sq = __dadd_rn(dist_sq, __dmul_rn(delta[k], delta[k]));
    const double dist = __dsqrt_rn(dist_sq);
    const double ds = __dadd_rn(dist, 0.01);
    spring = false;
    double target = 0.0;
    if (cell.pos | cell.neg) {
      target = cell.target;
      spring = (cell.pos && cell.neg) ? true : (cell.pos ? dist < target : dist > target);
    }
    if (spring) factor = __ddiv_rn(__dmul_rn(__dmul_rn(2.0, c.k), __dsub_rn(target, dist)), ds);
    else factor = __ddiv_rn(c.c_rep, __dmul_rn(__dmul_rn(__dmul_rn(2.0, ds), ds), ds));
  }
  static TL_D double norm(bool spring, double dp1, const Ctx& c) {
    return spring ? __dadd_rn(__dmul_rn(4.0, dp1), c.k) : dp1;
  }
  template <int D>
  static TL_D void pair(Point<D>& A, Point<D>& B, const Cell<double>& cell, const Ctx& c) {
    if (!(A.dp1 > 0.0 && B.dp1 > 0.0)) return;
    double delta[D];
#pragma unroll
    for (int k = 0; k < D; ++k) delta[k] = __dsub_rn(B.c[k], A.c[k]);
    bool spring; double factor;
    scalars<D>(delta, cell, c, spring, factor);
    const double nA = norm(spring, A.dp1, c), nB = norm(spring, B.dp1, c);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const double force = __dmul_rn(delta[k], factor);
      A.c[k] = __dsub_rn(A.c[k], __ddiv_rn(force, nA));
      B.c[k] = __dadd_rn(B.c[k], __ddiv_rn(force, nB));
    }
  }
  template <int D, int W_, bool kSum, bool kRotate>
  static TL_D void wave(Point<D> (&A)[kP], Point<D> (&B)[kP], const Cell<double> (&cell)[kP], const Ctx& c, int src) {
#pragma unroll
    for (int p = 0; p < kP; ++p) {
      const int q = kSum ? (W_ - p + kP) % kP : (p + W_) % kP;
      pair<D>(A[p], B[q], cell[p], c);
    }
    if (kRotate) {
#pragma unroll
      for (int q = 0; q < kP; ++q) B[q].shfl_from(src);
    }
  }
};

// ---------------------------------------------------------------------------------------
// Device helpers
// ---------------------------------------------------------------------------------------
TL_D unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// The caller's stop request (TileDev::abort, 16 readable bytes of mapped host memory) is fetched into shared memory by the
// bulk-copy unit at the start of an iteration and read at its end: nothing waits for the host round trip and no
// register holds the value across the pair passes.  One copy per iteration, so the barrier's phase is the parity of
// the copies issued before.
TL_D unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
TL_D void stop_word_init(unsigned long long* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
TL_D void stop_word_fetch(int* dst, unsigned long long* bar, const volatile int* src) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 16;" ::"r"(smem_u32(bar)) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 16, [%2];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(smem_u32(bar)) : "memory");
}
TL_D int stop_word_read(const int* s, unsigned long long* bar, unsigned parity) {
  unsigned done = 0;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
  return *reinterpret_cast<const volatile int*>(s);
}

// FitState moves between CTAs through L2 (never a stale L1 line).
static_assert(sizeof(FitState) % 8 == 0, "FitState is copied as 64-bit words");
TL_D void load_state(FitState& dst, const FitState* src) {
  unsigned long long* d = reinterpret_cast<unsigned long long*>(&dst);
  const unsigned long long* s = reinterpret_cast<const unsigned long long*>(src);
  for (int i = 0; i < (int)(sizeof(FitState) / 8); ++i) d[i] = __ldcg(s + i);
}
TL_D void store_state(FitState* dst, const FitState& src) {
  unsigned long long* d = reinterpret_cast<unsigned long long*>(dst);
  const unsigned long long* s = reinterpret_cast<const unsigned long long*>(&src);
  for (int i = 0; i < (int)(sizeof(FitState) / 8); ++i) __stcg(d + i, s[i]);
}

// A condition every lane of the warp agrees on, in a form the compiler can see is warp-uniform (a
// vote result): the pass functions below are compiled as convergent code only if every branch around
// their call sites is provably uniform.
TL_D bool warp_uniform(bool c) { return __all_sync(0xffffffffu, c); }

// Hand-off flags in shared memory (one per travelling tile).  Every lane polls the same word (one
// broadcast load), so the warp leaves the loop together: a single-lane spin would leave the warp
// diverged and every later shuffle would take the slow divergent path.
TL_D void wait_flag(volatile int* flag, int want) {
  while (!__all_sync(0xffffffffu, *flag >= want)) { }   // vote: a loop exit the compiler can see is uniform
  __threadfence_block();
  __syncwarp();
}
TL_D void post_flag(volatile int* flag, int value, int lane) {
  __syncwarp();
  __threadfence_block();
  if (lane == 0) *flag = value;
}

// Barrier across the G CTAs of one fit (all co-resident: cooperative launch).  Warp 0 arrives with
// one lane and then polls the generation word with all its lanes (uniform exit).
TL_D void gang_barrier(unsigned* bar, int G, unsigned& gen) {
  __syncthreads();
  if (G > 1) {
    if (threadIdx.x < 32) {
      unsigned last = 0u;
      if (threadIdx.x == 0) {
        __threadfence();
        last = (atomicAdd(&bar[0], 1u) == (unsigned)G - 1u) ? 1u : 0u;
        if (last) {
          atomicExch(&bar[0], 0u);
          __threadfence();
          atomicAdd(&bar[1], 1u);
        }
      }
      __syncwarp();
      while (ld_acquire_u32(&bar[1]) == gen) { __nanosleep(20); }
      __threadfence();
    }
    gen++;
    __syncthreads();
  }
}

// Round-to-round dependencies between the CTAs of a fit.  Every super-block takes part in exactly one
// task per cross round, so the task that uses super-block b in round r only has to wait for the task
// that used b in round r - 1 - not for the whole grid: done[b] counts the warps that have written
// their tile of b back (W per round), and a warp waits for r * W on both of its super-blocks.  Slack
// of a CTA then carries over to later rounds instead of being lost at a grid barrier per round.
TL_D void wait_blocks(const unsigned* done, int a, int b, unsigned want, int G) {
  if (G > 1) {
    while (ld_acquire_u32(done + a) < want || ld_acquire_u32(done + b) < want) { __nanosleep(20); }
    __syncwarp();
  }
}
TL_D void post_blocks(unsigned* done, int a, int b, int G, int lane) {
  if (G > 1) {
    __syncwarp();
    if (lane == 0) {
      __threadfence();
      atomicAdd(done + a, 1u);
      atomicAdd(done + b, 1u);
    }
  }
}
constexpr int kDoneOffset = 32;   // words of dv.barrier before the done[] counters (own cache lines)

template <int D>
struct TileShape {
  static constexpr int kReals = (D + 1) * kRow;    // D coordinate rows + the dp1 row, kTile slots each
};

// global AoS tile -> shared [k][65]
template <int D, class real>
TL_D void load_tile(real* s, const real* gpos, const real* gdp1, int tile, int lane) {
  if (tile < 0) {
#pragma unroll
    for (int k = 0; k <= D; ++k)
#pragma unroll
      for (int p = 0; p < kP; ++p) s[k * kRow + lane + 32 * p] = (real)0;
    return;
  }
  const real* base = gpos + (size_t)tile * (kTile * D);
#pragma unroll
  for (int j = 0; j < kP * D; ++j) {
    const int e = lane + 32 * j;
    s[(e % D) * kRow + (e / D)] = __ldcg(base + e);
  }
#pragma unroll
  for (int p = 0; p < kP; ++p) s[D * kRow + lane + 32 * p] = gdp1[(size_t)tile * kTile + lane + 32 * p];
}
template <int D, class real>
TL_D void store_tile(const real* s, real* gpos, int tile, int lane) {
  if (tile < 0) return;
  real* base = gpos + (size_t)tile * (kTile * D);
#pragma unroll
  for (int j = 0; j < kP * D; ++j) {
    const int e = lane + 32 * j;
    __stcg(base + e, s[(e % D) * kRow + (e / D)]);
  }
}

// Per-warp table of the measured pairs of one tile pair.  Combination c = kP * (A part) + (B part)
// (part p = slots 32p .. 32p+31 of a tile): tgt[c][step][lane], mask[c][kind][lane] with
// kind 0 = "pulls when closer than the target" (exact or '>'), 1 = "pulls when farther" (exact or '<').
// (Two 32-bit shared atomics per record: a 64-bit OR on shared memory is a compare-and-swap loop.)
constexpr int kCombos = kP * kP;
constexpr int kTableReals = kCombos * 32 * 32;
constexpr int kTableMasks = kCombos * 2 * 32;
template <class real>
struct WarpTable {
  real* tgt;
  uint32_t* mask;
};
struct LaneMasks {
  uint32_t pos[kCombos], neg[kCombos];
};

template <class real>
TL_D void table_clear(const WarpTable<real>& tb, int lane) {
#pragma unroll
  for (int j = 0; j < 2 * kCombos; ++j) tb.mask[j * 32 + lane] = 0u;
  __syncwarp();
}
template <class real>
TL_D void table_put(const WarpTable<real>& tb, int c, int idx, int lane_of, real target, int ty) {
  tb.tgt[(c * 32 + idx) * 32 + lane_of] = target;
  const uint32_t bit = 1u << idx;   // (selects instead of branches: nearly every record sets both masks)
  atomicOr(&tb.mask[(c * 2 + 0) * 32 + lane_of], ty != 2 ? bit : 0u);
  atomicOr(&tb.mask[(c * 2 + 1) * 32 + lane_of], ty != 1 ? bit : 0u);
}
template <class real>
TL_D LaneMasks table_masks(const WarpTable<real>& tb, int lane, bool filled) {
  LaneMasks m;
#pragma unroll
  for (int c = 0; c < kCombos; ++c) {
    m.pos[c] = filled ? tb.mask[(c * 2 + 0) * 32 + lane] : 0u;
    m.neg[c] = filled ? tb.mask[(c * 2 + 1) * 32 + lane] : 0u;
  }
  return m;
}
template <class real>
TL_D Cell<real> table_cell(const WarpTable<real>& tb, const LaneMasks& m, int c, int idx, int lane) {
  Cell<real> cell;
  const uint32_t bit = 1u << idx;
  cell.target = tb.tgt[(c * 32 + idx) * 32 + lane];   // garbage when not measured: discarded by the policy
  cell.pos = m.pos[c] & bit;
  cell.neg = m.neg[c] & bit;
  return cell;
}

// Scatter the measured pairs of bucket (lo, hi) into the warp's table.  `swap` = the A side is the
// higher-numbered tile.  Ring passes index by (combination, ring step, A lane).
// Warp-wide walk over edge records [beg, end): four independent 16-byte loads per lane are in flight
// before the first is used (the records come from L2 at best: one latency per 128 records, not four).
template <class F>
TL_D void for_each_edge(const EdgeRec* edges, uint32_t beg, uint32_t end, int lane, F&& fn) {
  for (uint32_t base = beg + lane; base < end; base += 128) {
    uint4 raw[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (base + 32 * k < end) raw[k] = __ldg(reinterpret_cast<const uint4*>(edges + base + 32 * k));
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (base + 32 * k < end) {
        EdgeRec r;
        r.target = __hiloint2double((int)raw[k].y, (int)raw[k].x);
        r.slot_lo = raw[k].z;
        r.slot_hi_type = raw[k].w;
        fn(r);
      }
  }
}
// Per-warp staging area for the edge records of the NEXT tile pass: filled by cp.async while the current
// pass runs, so that the scatter into the table reads shared memory instead of waiting for L2.
constexpr int kStage = 64 * kP;   // records per warp (a 1 %-dense 96 x 96 tile pair holds ~92); longer buckets
                                  // read their tail from global memory
TL_D void stage_issue(EdgeRec* stage, const EdgeRec* edges, uint32_t beg, uint32_t end, int lane) {
  const uint32_t n = min(end - beg, (uint32_t)kStage);
  for (uint32_t i = lane; i < n; i += 32) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(stage + i);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(edges + beg + i) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}
TL_D void stage_wait() {
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
}
template <class F>
TL_D void for_each_staged(const EdgeRec* stage, uint32_t count, int lane, F&& fn) {
  for (uint32_t i = lane; i < count; i += 32) fn(stage[i]);
}

// (Called by the kernel right before the pass function: the pass loops keep their register allocation
// to themselves.)  The first min(end - beg, kStage) records are read from `stage` when it is not null.
template <class real>
TL_D void fill_table_ring(const WarpTable<real>& tb, const EdgeRec* edges, const EdgeRec* stage, uint32_t beg,
                          uint32_t end, bool swap, const RingParams& rp, int lane) {
  if (beg == end) return;   // warp-uniform
  table_clear<real>(tb, lane);
  auto put = [&](const EdgeRec& r) {
    const int lo = (int)(r.slot_lo % kTile), hi = (int)((r.slot_hi_type & 0x3fffffffu) % kTile);
    const int ty = r.slot_hi_type >> 30;
    const int a = swap ? hi : lo, b = swap ? lo : hi;
    const int la = a & 31, lb = b & 31;
    table_put<real>(tb, kP * (a >> 5) + (b >> 5), ring_step(rp, la, lb), la, (real)r.target, ty);
  };
  const uint32_t ns = stage ? min(end - beg, (uint32_t)kStage) : 0u;
  for_each_staged(stage, ns, lane, put);
  for_each_edge(edges, beg + ns, end, lane, put);
}
// Intra passes index by (combination seen from the lane, xor distance, lane); pairs among a lane's
// own kP slots sit at index 0 (xor distance 0 never occurs otherwise).
template <class real>
TL_D void fill_table_xor(const WarpTable<real>& tb, const EdgeRec* edges, uint32_t beg, uint32_t end, int lane) {
  if (beg == end) return;
  table_clear<real>(tb, lane);
  for_each_edge(edges, beg, end, lane, [&](const EdgeRec& r) {
    const int u = (int)(r.slot_lo % kTile), v = (int)((r.slot_hi_type & 0x3fffffffu) % kTile);
    const int ty = r.slot_hi_type >> 30;
    const int lu = u & 31, lv = v & 31, pu = u >> 5, pv = v >> 5;
    const int x = lu ^ lv;
    if (x == 0) {
      table_put<real>(tb, kP * pu + pv, 0, lu, (real)r.target, ty);   // pu < pv
    } else {
      table_put<real>(tb, kP * pu + pv, x, lu, (real)r.target, ty);
      table_put<real>(tb, kP * pv + pu, x, lv, (real)r.target, ty);
    }
  });
}

TL_D void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Bucket range of tile pair (ta, tb) and an L2 prefetch of its edge records (issued one task ahead
// of use: the edge stream is far larger than L2, the per-pass loads must not go to DRAM).
TL_D uint2 bucket_range(const uint32_t* bucket_off, const EdgeRec* edges, int T, int ta, int tb) {
  const int lo = ta < tb ? ta : tb, hi = ta < tb ? tb : ta;
  const size_t key = (size_t)lo * T + hi;
  uint2 r;
  r.x = bucket_off[key];
  r.y = bucket_off[key + 1];
  const char* p = reinterpret_cast<const char*>(edges + r.x);
  const char* e = reinterpret_cast<const char*>(edges + r.y);
  for (int i = 0; i < 16 && p < e; ++i, p += 128) prefetch_l2(p);
  return r;
}

// Compile-time loop over the kP waves of one step.
template <int D, class M, bool kSum, int W_ = 0>
struct Waves {
  typedef typename M::real real;
  static TL_D void run(typename M::template Point<D> (&A)[kP], typename M::template Point<D> (&B)[kP],
                       const WarpTable<real>& tb, const LaneMasks& m, int idx, int lane, const typename M::Ctx& ctx,
                       int src) {
    Cell<real> cell[kP];
#pragma unroll
    for (int p = 0; p < kP; ++p) {
      const int q = kSum ? (W_ - p + kP) % kP : (p + W_) % kP;
      cell[p] = table_cell<real>(tb, m, kP * p + q, idx, lane);
    }
    M::template wave<D, W_, kSum, !kSum && W_ == kP - 1>(A, B, cell, ctx, src);   // ring pass: rotate B in the last wave
    Waves<D, M, kSum, W_ + 1>::run(A, B, tb, m, idx, lane, ctx, src);
  }
};
template <int D, class M, bool kSum>
struct Waves<D, M, kSum, kP> {
  typedef typename M::real real;
  static TL_D void run(typename M::template Point<D> (&)[kP], typename M::template Point<D> (&)[kP],
                       const WarpTable<real>&, const LaneMasks&, int, int, const typename M::Ctx&, int) {}
};

// tile A x tile B (kTile x kTile pairs), 32 ring steps of kP waves of kP pair visits per lane.  Lane a
// keeps A[p] = slot a + 32p; the travelling B[q] = slot b + 32q with b = ring_b(a, i).  Wave w of a step
// pairs A[p] with B[(p + w) % kP]: kP independent visits, a perfect matching over the warp.
//
// A function of its own on purpose (not inlined, arguments by value): inside the kernel the compiler
// cannot prove that a warp is converged where the pass is called (the conditions around it are loaded
// from shared memory) and guards every group of shuffles with a divergence check (BRA.DIV) which
// nothing can be scheduled across; a function body is compiled as convergent code, so the shuffles
// issue between the FMAs.  The callers guarantee convergence (warp-uniform branches, __syncwarp).
template <int D, class M>
__device__ __noinline__ void ring_pass(typename M::real* sA, typename M::real* sB, RingParams rp, bool filled,
                                       const WarpTable<typename M::real>& tb, const typename M::Ctx& ctx, int lane) {
  typedef typename M::real real;
  const LaneMasks m = table_masks<real>(tb, lane, filled);
  typename M::template Point<D> A[kP], B[kP];
  const int b0 = (lane + rp.s0) & 31;
#pragma unroll
  for (int p = 0; p < kP; ++p) { A[p].load(sA, lane + 32 * p, ctx); B[p].load(sB, b0 + 32 * p, ctx); }
  const int src = (lane + rp.g) & 31;
#pragma unroll kRingUnroll
  for (int i = 0; i < 32; ++i) {
    // the last wave of every step hands the B points on (also after step 31: that rotation brings every
    // B point back to the lane that loaded it)
    Waves<D, M, false>::run(A, B, tb, m, i, lane, ctx, src);
  }
  const int bf = b0;
#pragma unroll
  for (int p = 0; p < kP; ++p) { A[p].store(sA, lane + 32 * p); B[p].store(sB, bf + 32 * p); }
}

// tile x itself.  Lane a owns S[p] = slot a + 32p: first the pairs among its own slots, then 31 XOR
// steps against lane a^x.  Wave w of a step visits (S[p], O[(w - p) mod kP]) - the same set of pairs
// seen from either lane - two-sided on the lane's local copies O of the partner's points, which the
// partner updates identically for itself.
template <int D, class M>
__device__ __noinline__ void intra_pass(typename M::real* sT, XorParams xp, bool filled,
                                        const WarpTable<typename M::real>& tb, const typename M::Ctx& ctx, int lane) {
  typedef typename M::real real;
  const LaneMasks m = table_masks<real>(tb, lane, filled);
  typename M::template Point<D> S[kP], O[kP];
#pragma unroll
  for (int p = 0; p < kP; ++p) S[p].load(sT, lane + 32 * p, ctx);
#pragma unroll
  for (int p = 0; p < kP; ++p)
#pragma unroll
    for (int q = p + 1; q < kP; ++q) M::template pair<D>(S[p], S[q], table_cell<real>(tb, m, kP * p + q, 0, lane), ctx);
#pragma unroll 1
  for (int i = 0; i < 31; ++i) {
    const int x = xor_at(xp, i);
#pragma unroll
    for (int p = 0; p < kP; ++p) O[p].shfl_xor_of(S[p], x);
    Waves<D, M, true>::run(S, O, tb, m, x, lane, ctx, 0);
  }
#pragma unroll
  for (int p = 0; p < kP; ++p) S[p].store(sT, lane + 32 * p);
}

// One point's coordinates from global memory (through L2: other CTAs wrote them), 128-bit loads when
// the row size allows.
template <int D, class real>
TL_D void load_row(const real* p, real (&out)[D]) {
  constexpr int kVec = 16 / (int)sizeof(real);
  if ((D % kVec) == 0) {
#pragma unroll
    for (int j = 0; j < D / kVec; ++j) {
      const uint4 v = __ldcg(reinterpret_cast<const uint4*>(p) + j);
      if (sizeof(real) == 4) {
        out[4 * j + 0] = (real)__uint_as_float(v.x); out[4 * j + 1] = (real)__uint_as_float(v.y);
        out[4 * j + 2] = (real)__uint_as_float(v.z); out[4 * j + 3] = (real)__uint_as_float(v.w);
      } else {
        out[2 * j + 0] = (real)__hiloint2double((int)v.y, (int)v.x);
        out[2 * j + 1] = (real)__hiloint2double((int)v.w, (int)v.z);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < D; ++j) out[j] = __ldcg(p + j);
  }
}

// One edge's term of the MAE (src/optimization.cpp:62-76): |target - dist| of a measured pair, and of a
// threshold pair only while the threshold is violated.  `raw` is the 16-byte EdgeRec.
template <int D, class real>
TL_D void edge_error(const uint4& raw, const real (&ra)[D], const real (&rb)[D], double& e_sum, double& e_cnt) {
  const double target = __hiloint2double((int)raw.y, (int)raw.x);
  const int ty = raw.w >> 30;
  double ss = 0.0;
  if (sizeof(real) == 8) {   // exact policy: the reference's operations, one rounding each
#pragma unroll
    for (int j = 0; j < D; ++j) {
      const double df = __dsub_rn((double)rb[j], (double)ra[j]);
      ss = __dadd_rn(ss, __dmul_rn(df, df));
    }
  } else {                   // FP32 positions: difference in FP32 (exact for nearby coordinates), squares summed in FP64
#pragma unroll
    for (int j = 0; j < D; ++j) {
      const double df = (double)(rb[j] - ra[j]);
      ss = fma(df, df, ss);
    }
  }
  const double dist = __dsqrt_rn(ss);
  const bool contributes = (ty == 0) || (ty == 1 && dist < target) || (ty == 2 && dist > target);
  if (contributes) { e_sum += fabs(target - dist); e_cnt += 1.0; }
}

// This thread's edges e0, e0 + stride, ... in batches of K with every load of a batch issued before its
// first use; stops (and leaves e0) where fewer than K edges remain.
template <int D, class real, int K>
TL_D void edge_batches(const TileDev<real>& dv, long long& e0, long long stride, double& e_sum, double& e_cnt) {
  for (; e0 + (K - 1) * stride < dv.n_edges; e0 += stride * K) {
    uint4 raw[K];
#pragma unroll
    for (int k = 0; k < K; ++k) raw[k] = __ldcs(reinterpret_cast<const uint4*>(dv.edges + e0 + k * stride));
    real ra[K][D], rb[K][D];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      load_row<D, real>(dv.pos + (size_t)raw[k].z * D, ra[k]);
      load_row<D, real>(dv.pos + (size_t)(raw[k].w & 0x3fffffffu) * D, rb[k]);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) edge_error<D, real>(raw[k], ra[k], rb[k], e_sum, e_cnt);
  }
}

// Deterministic CTA reduction of (sum, count, flag); result valid in thread 0.
TL_D void block_reduce3(double& a, double& b, double& c, double* scratch /* [3*32] */) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_down_sync(full, a, o);
    b += __shfl_down_sync(full, b, o);
    c += __shfl_down_sync(full, c, o);
  }
  if (lane == 0) { scratch[warp] = a; scratch[32 + warp] = b; scratch[64 + warp] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    a = 0; b = 0; c = 0;
    for (int w = 0; w < nw; ++w) { a += scratch[w]; b += scratch[32 + w]; c += scratch[64 + w]; }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------
// The persistent loop: up to n_iters iterations of one fit, run by G CTAs of W warps (`cta` = this
// CTA's index among them).
// ---------------------------------------------------------------------------------------
template <int D, class M>
TL_D void tile_body(const TileDev<typename M::real>& dv, const Geometry& geo, const FitParams& prm, int n_iters,
                    volatile int* host_flag, const int cta) {
  typedef typename M::real real;
  constexpr int TS = TileShape<D>::kReals;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ FitState st;
  __shared__ double red_scratch[96];
  __shared__ unsigned long long s_key[kIterKeys];   // iter_key(geo, iter, salt) of the running iteration

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = geo.W;
  real* s_tiles = reinterpret_cast<real*>(smem_raw);
  real* s_tgt = s_tiles + (size_t)2 * W * TS;
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_tgt + (size_t)W * kTableReals);
  int* s_tid = reinterpret_cast<int*>(s_mask + W * kTableMasks);
  int* s_flag = s_tid + 2 * W;
  EdgeRec* s_stage_all = reinterpret_cast<EdgeRec*>((reinterpret_cast<uintptr_t>(s_flag + W) + 15) & ~(uintptr_t)15);
  EdgeRec* s_stage = s_stage_all + warp * kStage;
  // this iteration's tile placement and round order (geo.table): [side-0 slots][side-1 slots][rounds]
  int* s_perm = reinterpret_cast<int*>(s_stage_all + W * kStage);
  const int n_side0 = perm_table_side0(geo), n_slots = geo.S * W;
  auto tile_of = [&](int slot, int side) {
    return geo.table ? s_perm[(side ? n_side0 : 0) + slot] : tile_at_k(geo, s_key[side ? 7 : 1], slot, side);
  };
  const WarpTable<real> tb{s_tgt + (size_t)warp * kTableReals, s_mask + warp * kTableMasks};

  __shared__ __align__(16) int s_stop_word[4];
  __shared__ __align__(8) unsigned long long s_stop_bar;

  unsigned gen = 0;
  if (tid == 0) load_state(st, dv.state);
  // Only CTA 0 reads the stop request (the CTAs of a fit must agree), and a stop never overrides a fit that has already
  // ended.  A CTA or chunk that starts after the request runs no iteration.
  if (cta == 0 && tid == 0 && dv.abort) {
    stop_word_init(&s_stop_bar);
    if (*dv.abort && !st.stop && st.iter < prm.n_iter) { st.stop = 1; st.status = kStatusStopped; }
  }
  if (geo.G > 1) gen = ld_acquire_u32(&dv.barrier[1]);
  __syncthreads();
  unsigned* done = dv.barrier + kDoneOffset;
  unsigned epoch = 0;   // cross rounds completed since the start of this launch
  if (geo.G > 1) {
    for (int b = cta * blockDim.x + tid; b < geo.S; b += geo.G * blockDim.x) __stcg(done + b, 0u);
    if (dv.abort && cta == 0 && tid == 0) store_state(dv.state, st);   // publish CTA 0's decision
    gang_barrier(dv.barrier, geo.G, gen);
    if (dv.abort) {
      if (cta != 0 && tid == 0) load_state(st, dv.state);
      __syncthreads();
    }
  }

  for (int it = 0; it < n_iters; ++it) {
    if (st.stop || st.iter >= prm.n_iter) break;   // never past n_iter: trace[] holds n_iter entries, the forced last check is iter == n_iter - 1
    const int iter = st.iter;
    if (cta == 0 && tid == 0 && dv.abort && geo.do_end) stop_word_fetch(s_stop_word, &s_stop_bar, dv.abort);
    const typename M::Ctx ctx = M::make_ctx(st.k, prm.c_repulsion);
    if (tid < kIterKeys) s_key[tid] = iter_key(geo, iter, (uint32_t)tid);
    if (geo.table) {
      const uint64_t k1 = iter_key(geo, iter, 1u), k7 = iter_key(geo, iter, 7u), k2 = iter_key(geo, iter, 2u);
      for (int i = tid; i < n_slots; i += blockDim.x)
        s_perm[i] = i < n_side0 ? tile_at_k(geo, k1, i, 0) : tile_at_k(geo, k7, i - n_side0, 1);
      for (int r = tid; r < cross_rounds(geo); r += blockDim.x) s_perm[n_slots + r] = round_at_k(geo, k2, r);
    }
    __syncthreads();

    // ---------------- cross rounds ----------------
    for (int r = 0; r < cross_rounds(geo); ++r) {
      const int rr = geo.table ? s_perm[n_slots + r] : round_at_k(geo, s_key[2], r);
      for (int tt = 0; tt < geo.m; ++tt) {
        int X, Y;
        cross_task(geo, rr, cta * geo.m + tt, X, Y);
        const int tX = tile_of(X * W + warp, 0), tY = tile_of(Y * W + warp, geo.kind);
        const int bX = X, bY = geo.kind == 1 ? geo.S / 2 + Y : Y;   // counters: the two sides of a bipartite job apart
        wait_blocks(done, bX, bY, epoch * (unsigned)W, geo.G);
        if (lane == 0) { s_tid[warp] = tX; s_tid[W + warp] = tY; s_flag[warp] = 0; }
        load_tile<D, real>(s_tiles + (size_t)warp * TS, dv.pos, dv.dp1, tX, lane);
        load_tile<D, real>(s_tiles + (size_t)(W + warp) * TS, dv.pos, dv.dp1, tY, lane);
        __syncthreads();
        const int rot = cross_rot_k(geo, s_key[5], X, Y);
        // lane v fetches the bucket range of this warp's sub-round v and prefetches its records
        uint2 my_rng = make_uint2(0u, 0u);
        if (lane < W) {
          const int tA = s_tid[warp], tB = s_tid[W + (warp + lane + rot) % W];
          if (tA >= 0 && tB >= 0) my_rng = bucket_range(dv.bucket_off, dv.edges, geo.T, tA, tB);
        }
        stage_issue(s_stage, dv.edges, __shfl_sync(0xffffffffu, my_rng.x, 0), __shfl_sync(0xffffffffu, my_rng.y, 0), lane);
        // Sub-rounds without a CTA barrier: tile Y[b] is handed from warp to warp.  s_flag[b] counts
        // the passes completed on Y[b]; the pass of sub-round v needs exactly v of them (the one
        // before it ran on warp + 1), so the waits form chains that end at sub-round 0.
        for (int v = 0; v < W; ++v) {
          const int bw = (warp + v + rot) % W;
          const int tA = s_tid[warp], tB = s_tid[W + bw];
          const uint32_t beg = __shfl_sync(0xffffffffu, my_rng.x, v), end = __shfl_sync(0xffffffffu, my_rng.y, v);
          const int vn = v + 1 < W ? v + 1 : v;
          const uint32_t nbeg = __shfl_sync(0xffffffffu, my_rng.x, vn), nend = __shfl_sync(0xffffffffu, my_rng.y, vn);
          wait_flag(s_flag + bw, v);
          const bool live = warp_uniform(tA >= 0 && tB >= 0);
          const RingParams rp = ring_params_k(s_key[3], tA, tB);
          stage_wait();
          if (live) fill_table_ring<real>(tb, dv.edges, s_stage, beg, end, tA > tB, rp, lane);
          __syncwarp();
          if (v + 1 < W) stage_issue(s_stage, dv.edges, nbeg, nend, lane);   // records of the next sub-round, in flight during this pass
          if (live)
            ring_pass<D, M>(s_tiles + (size_t)warp * TS, s_tiles + (size_t)(W + bw) * TS, rp, beg != end, tb, ctx, lane);
          post_flag(s_flag + bw, v + 1, lane);
        }
        wait_flag(s_flag + warp, W);   // every pass on Y[warp] is done: this warp writes it back
        store_tile<D, real>(s_tiles + (size_t)warp * TS, dv.pos, tX, lane);
        store_tile<D, real>(s_tiles + (size_t)(W + warp) * TS, dv.pos, tY, lane);
        post_blocks(done, bX, bY, geo.G, lane);
      }
      ++epoch;
    }

    // ---------------- diagonal round (kind 0 only) ----------------
    for (int tt = 0; tt < (geo.kind == 0 ? geo.m : 0); ++tt) {
      const int q = cta * geo.m + tt;
      const int tX = tile_of((2 * q) * W + warp, 0), tY = tile_of((2 * q + 1) * W + warp, 0);
      wait_blocks(done, 2 * q, 2 * q + 1, epoch * (unsigned)W, geo.G);
      if (lane == 0) { s_tid[warp] = tX; s_tid[W + warp] = tY; }
      load_tile<D, real>(s_tiles + (size_t)warp * TS, dv.pos, dv.dp1, tX, lane);
      load_tile<D, real>(s_tiles + (size_t)(W + warp) * TS, dv.pos, dv.dp1, tY, lane);
      __syncthreads();
      const int Mt = diag_subrounds(W), rot = diag_rot_k(geo, s_key[6], q);
      // lanes 0..Mt-1: bucket of this warp's tile pair in sub-round `lane`; lanes 16, 17: own tiles
      uint2 my_rng = make_uint2(0u, 0u);
      {
        int ta = -1, tb2 = -1;
        if (lane < Mt) {
          int sb, ia, ib;
          if (diag_pair(W, lane, rot, warp, sb, ia, ib)) { ta = s_tid[sb * W + ia]; tb2 = s_tid[sb * W + ib]; }
        } else if (lane == 16) { ta = tb2 = tX; }
        else if (lane == 17) { ta = tb2 = tY; }
        if (ta >= 0 && tb2 >= 0) my_rng = bucket_range(dv.bucket_off, dv.edges, geo.T, ta, tb2);
      }
      for (int u = 0; u < Mt; ++u) {
        int sb, ia, ib;
        const uint32_t beg = __shfl_sync(0xffffffffu, my_rng.x, u), end = __shfl_sync(0xffffffffu, my_rng.y, u);
        if (warp_uniform(diag_pair(W, u, rot, warp, sb, ia, ib))) {
          const int tA = s_tid[sb * W + ia], tB = s_tid[sb * W + ib];
          if (warp_uniform(tA >= 0 && tB >= 0)) {
            const RingParams rp = ring_params_k(s_key[3], tA, tB);
            fill_table_ring<real>(tb, dv.edges, nullptr, beg, end, tA > tB, rp, lane);
            __syncwarp();
            ring_pass<D, M>(s_tiles + (size_t)(sb * W + ia) * TS, s_tiles + (size_t)(sb * W + ib) * TS, rp, beg != end,
                            tb, ctx, lane);
          }
        }
        __syncthreads();
      }
      {
        const uint32_t bx = __shfl_sync(0xffffffffu, my_rng.x, 16), ex = __shfl_sync(0xffffffffu, my_rng.y, 16);
        const uint32_t by = __shfl_sync(0xffffffffu, my_rng.x, 17), ey = __shfl_sync(0xffffffffu, my_rng.y, 17);
        if (warp_uniform(tX >= 0)) {
          fill_table_xor<real>(tb, dv.edges, bx, ex, lane);
          __syncwarp();
          intra_pass<D, M>(s_tiles + (size_t)warp * TS, xor_params_k(s_key[4], tX), bx != ex, tb, ctx, lane);
        }
        if (warp_uniform(tY >= 0)) {
          fill_table_xor<real>(tb, dv.edges, by, ey, lane);
          __syncwarp();
          intra_pass<D, M>(s_tiles + (size_t)(W + warp) * TS, xor_params_k(s_key[4], tY), by != ey, tb, ctx, lane);
        }
      }
      store_tile<D, real>(s_tiles + (size_t)warp * TS, dv.pos, tX, lane);
      store_tile<D, real>(s_tiles + (size_t)(W + warp) * TS, dv.pos, tY, lane);
      __syncwarp();
    }
    gang_barrier(dv.barrier, geo.G, gen);

    if (!geo.do_end) continue;   // a job of a sharded iteration: the end phase is a launch of its own

    // ---------------- end of iteration: cooling, MAE, controller, finite check ----------------
    const bool check = is_check_iter(iter, prm);
    const bool fin = ((iter + 1) % 10 == 0);
    if (tid == 0) {
      st.k = st.k * (1.0 - prm.cooling_rate);
      st.pair_updates += dv.pairs_per_iter;
    }
    if (check || fin) {
      double e_sum = 0.0, e_cnt = 0.0, bad = 0.0;
      if (check) {
        // Edge MAE (src/optimization.cpp:54-81): kEB edges per thread and trip, every load of the batch
        // issued before the first use - the CTAs of the pair loop are all the threads there are, so the
        // memory parallelism has to come from inside a thread.
        constexpr int kEB = sizeof(real) == 4 ? (D <= 8 ? 8 : 4) : 2;   // ~128 registers of row data
        const long long stride = (long long)geo.G * blockDim.x;
        long long e0 = (long long)cta * blockDim.x + tid;
        edge_batches<D, real, kEB>(dv, e0, stride, e_sum, e_cnt);
        if (kEB > 2) edge_batches<D, real, 2>(dv, e0, stride, e_sum, e_cnt);   // short lists: keep the tail parallel too
        edge_batches<D, real, 1>(dv, e0, stride, e_sum, e_cnt);
      }
      if (fin) {
        const size_t total = (size_t)geo.T * kTile * D;
        for (size_t x = (size_t)cta * blockDim.x + tid; x < total; x += (size_t)geo.G * blockDim.x)
          if (!isfinite((double)__ldcg(dv.pos + x))) bad = 1.0;
      }
      block_reduce3(e_sum, e_cnt, bad, red_scratch);
      if (tid == 0) {
        double* p = dv.partials + (size_t)cta * 4;
        __stcg(p, e_sum); __stcg(p + 1, e_cnt); __stcg(p + 2, bad);
      }
      gang_barrier(dv.barrier, geo.G, gen);
      if (cta == 0 && tid == 0) {
        double s = 0.0, c = 0.0, b = 0.0;
        for (int g = 0; g < geo.G; ++g) {
          const double* p = dv.partials + (size_t)g * 4;
          s += __ldcg(p); c += __ldcg(p + 1); b += __ldcg(p + 2);
        }
        st.snapshot = 0;
        if (check) {
          controller_check(st, prm, iter, s, (long long)c);
          if (dv.trace) dv.trace[iter] = st.last_error;
        }
        if (!st.stop && fin && b > 0.0) { st.status = 2; st.fail_iter = iter + 1; st.stop = 1; }
        st.iter = iter + 1;
        if (dv.abort && stop_word_read(s_stop_word, &s_stop_bar, it & 1) && !st.stop && st.iter < prm.n_iter) {
          st.stop = 1; st.status = kStatusStopped;
        }
        store_state(dv.state, st);
      }
      gang_barrier(dv.barrier, geo.G, gen);
      if (cta != 0 && tid == 0) load_state(st, dv.state);
      __syncthreads();
      if (st.snapshot) {
        const size_t total = (size_t)geo.T * kTile * D;
        for (size_t x = (size_t)cta * blockDim.x + tid; x < total; x += (size_t)geo.G * blockDim.x)
          dv.best[x] = __ldcg(dv.pos + x);
        gang_barrier(dv.barrier, geo.G, gen);
      }
    } else {
      if (tid == 0) {
        st.iter = iter + 1;
        // (every fetch is waited for; a fit of several CTAs stops only where CTA 0 publishes its state, above)
        if (cta == 0 && dv.abort && stop_word_read(s_stop_word, &s_stop_bar, it & 1) && geo.G == 1 && !st.stop &&
            st.iter < prm.n_iter) {
          st.stop = 1; st.status = kStatusStopped;
        }
      }
      __syncthreads();
    }
  }
  if (cta == 0 && tid == 0) {
    store_state(dv.state, st);
    if (host_flag) { host_flag[1] = st.iter; __threadfence_system(); host_flag[0] = st.stop; }
  }
}

// One fit per launch: G CTAs (co-operative launch when G > 1).
template <int D, class M>
__global__ void __launch_bounds__(M::kMaxWarps * 32, 1)
tile_kernel(TileDev<typename M::real> dv, Geometry geo, FitParams prm, int n_iters, volatile int* host_flag) {
  tile_body<D, M>(dv, geo, prm, n_iters, host_flag, (int)blockIdx.x);
}

// Many fits per launch, one CTA each (the CV grid): CTA b runs jobs[b].  All jobs of a launch have the
// same D, precision and W; fits that have already stopped return at once.
template <int D, class M>
__global__ void __launch_bounds__(M::kMaxWarps * 32, 1)
tile_batch_kernel(const BatchJob<typename M::real>* __restrict__ jobs) {
  typedef BatchJob<typename M::real> Job;
  __shared__ Job job;
  static_assert(sizeof(Job) % 4 == 0, "BatchJob is copied as 32-bit words");
  const uint32_t* src = reinterpret_cast<const uint32_t*>(jobs + blockIdx.x);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&job);
  for (int i = threadIdx.x; i < (int)(sizeof(Job) / 4); i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  tile_body<D, M>(job.dv, job.geo, job.prm, job.n_iters, job.host_flag, 0);
}

}  // namespace TL_PNS
}  // namespace tl
