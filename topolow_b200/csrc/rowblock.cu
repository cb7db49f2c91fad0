// topolow_b200/csrc/rowblock.cu
//
// Row-block ("owner computes") mode of the embedding loop - the partitioning of one large map that
// SURVEY.md section 8e / BASELINE.json's north_star describe: the points are cut into G contiguous row
// blocks, GPU g owns the updates of its rows and computes them against a replica of ALL positions;
// within an iteration a point's own springs are applied one after another (Gauss-Seidel along the row),
// other points are read at their position of the iteration's start (Jacobi across points and across
// GPUs); the new rows are stored straight into every replica over NVLink (peer stores) and one
// flag exchange per iteration is the only synchronisation.  G = 1 is the same code on one GPU.
//
// One iteration on the replica P of all positions (reference: /root/reference/src/optimization.cpp):
//   repulse_kernel  R_i = -sum_{j != i} (P_j - P_i) * c / (2 (|P_j - P_i| + 0.01)^3) / (deg_i + 1)   (:269-281
//                   seen from i's side), a tiled one-sided N-body pass in packed FP32: a work item is
//                   256 own rows x one chunk of 2048 partners streamed through shared memory by cp.async.
//   spring_kernel   x = P_i, then for every measured pair (i, j) of row i in turn (:226-256, i's side):
//                   spring iff exact, or '>' and dist < target, or '<' and dist > target (:237-243);
//                   x -= (P_j - x) * 2k (target - dist) / (dist + 0.01) / (4 (deg_i + 1) + k)  (:246-253) and the
//                   repulsion R_i contains for this pair is taken back (a pair in spring state is not
//                   repelled); a satisfied threshold keeps its repulsion (:257-267).  One thread per row, records
//                   in degree-padded slices of 32 rows (SELL-32) so that a warp's record loads are one contiguous
//                   256-byte line.  Runs on a second stream NEXT TO the repulsion pass (both read only P).
//   combine_kernel  P'_i = x + R_i goes to every replica (peer stores), cooling (:289), one flag per peer.
//   mae_kernel      on check iterations: sum |target - dist| and count over the measured pairs that are exact
//                   or violated (:54-81) on P', FP64 sums, fixed summation tree; partial sums go to every replica.
//   ctl_kernel      cooling happened in the spring kernel (:289); three-way controller with best-state snapshot
//                   (:303-357, common.cuh::controller_check), finite check every 10 iterations (:359-361).
// Every unordered pair is visited once from each side per iteration and each side moves only its own
// endpoint, by what the reference's visit of the pair would move it.  Results do not depend on G (the
// summation trees are fixed), which is what the tests check; the scheme is compared with the reference's
// sequential loop statistically (tests/test_gpu_rowblock.py) and with its own CPU restatement
// (oracle/relaxed_oracle.cpp) numerically.
#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstring>
#include <functional>
#include <memory>
#include <thread>
#include <vector>

#include "plan.h"
#include "rowblock.h"

namespace tl {

std::vector<int32_t> random_permutation(int64_t n, uint64_t seed);   // plan.cu

namespace {

constexpr uint64_t kRowLayoutSeed = 0x726f77626c6f636bULL;
constexpr int kStageJ = 128;   // partners per shared-memory stage
constexpr int kStages = 3;
constexpr int kFlagStride = 32;   // 32-bit words between the flag words of two ranks (128 bytes)
constexpr int kWalkRegs = 112;    // register cap of spring_kernel (see there)
constexpr int kWalkRegsWide = 168;   // ... for ndim 17..32 (H > 8), which never runs beside the two-GEMM pass
constexpr int kRepUnrollWide = 1, kRepRegsWide = 128;   // repulse_kernel for ndim 17..32: partner unroll, register cap
constexpr unsigned long long kWaitNs = 20ull * 1000ull * 1000ull * 1000ull;

struct RowDev {
  int n, slots, D, Dp, G, rank, row0, rows, chunks;
  int rparts;                        // partial-sum entries per row in rpart: chunks (2 x chunks for the tensor-core pass)
  int adaptive;                      // 1: the repulsion form is chosen per iteration on the device (counters[6], set by image_tc_kernel)
  int series;                        // tensor form: weights by the one-MUFU series where the probe allows it (adaptive) / always (not adaptive)
  int probe_k;                       // sampled partners per row of the near-pair probe
  unsigned probe_limit;              // tensor form while the probe finds at most this many near pairs
  int no_wait;                       // measurement only (TOPOLOW_IGNORE_PEERS): one rank of a sharded map timed without its peers
  unsigned long long cap_rows;       // rows of one position buffer (slots rounded up to a chunk)
  float* pos[kMaxShards];            // replica q: [2][cap_rows][Dp]
  double* red[kMaxShards];           // replica q: [slots / 128][4]  {sum |err|, count, non-finite, -}
  unsigned* flags[kMaxShards];       // replica q: [kMaxShards][kFlagStride], word r = epoch reached by rank r
  float* best;                       // [cap_rows][Dp]
  const float* dp1;                  // [slots] degree + 1 (0 = padding row)
  float* rpart;                      // [chunks][rows][Dp] repulsion sums per partner chunk
  float* xs;                         // [rows][Dp] positions of the own rows after the spring walk (before the repulsion is added)
  float centre[16];                  // centroid of the initial positions (fixed for the fit, the same on every rank)
  const uint2* recs;                 // spring records of the own rows, SELL-32: {partner | type << 30, target}
  const unsigned long long* soff;    // [rows / 32] first record of a slice
  const int* swidth;                 // [rows / 32] records per row of a slice
  const uint2* mrecs;                // the records this rank counts in the MAE (every pair once over all ranks)
  const unsigned long long* moff;
  const int* mwidth;
  FitState* state;
  double* trace;
  unsigned* counters;                // [0..2] tickets of the "last CTA" of a launch / work items; [3], [4] near pairs the probe found (series
                                     // form / plain), [5] its ticket, [6] form of this iteration (0 FP32, 1 tensor, 2 tensor with the series
                                     // weights), [7] iterations run in a tensor form
  volatile int* host_flag;           // mapped: [0] stop, [1] iterations done
  unsigned long long pairs_per_iter;
  unsigned long long seed;
};

typedef void (*RepulseFn)(RowDev, int, unsigned);

// Adaptive runs launch both repulsion kernels every iteration; the one whose form was not chosen returns at once.
TL_D bool form_is_tensor(const RowDev& dv) { return __ldcg(&dv.counters[6]) != 0u; }

// ---------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------
TL_D float sqrt_approx(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
TL_D float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
TL_D unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
TL_D void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
TL_D unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
TL_D void cp_async16(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
TL_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> TL_D void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Rows are stored with a stride of kStride<H> floats (a multiple of 4: every row starts on a 16-byte boundary,
// odd H leaves two pad floats that are never computed on).
template <int H> struct Row { static constexpr int kStride = (2 * H + 3) / 4 * 4; };

// H packed pairs of one point from (shared or global) memory: 16-byte loads, one 8-byte tail when H is odd.
template <int H>
TL_D void ld_point(const float* __restrict__ p, float2 (&v)[H]) {
#pragma unroll
  for (int k = 0; k < H / 2; ++k) {
    const float4 t = reinterpret_cast<const float4*>(p)[k];
    v[2 * k] = make_float2(t.x, t.y); v[2 * k + 1] = make_float2(t.z, t.w);
  }
  if constexpr (H % 2 == 1) v[H - 1] = reinterpret_cast<const float2*>(p)[H - 1];
}
template <int H>
TL_D void st_point(float* __restrict__ p, const float2 (&v)[H]) {
#pragma unroll
  for (int k = 0; k < H / 2; ++k)
    reinterpret_cast<float4*>(p)[k] = make_float4(v[2 * k].x, v[2 * k].y, v[2 * k + 1].x, v[2 * k + 1].y);
  if constexpr (H % 2 == 1) reinterpret_cast<float2*>(p)[H - 1] = v[H - 1];
}

// |q + np|^2 (np = -p); delta is kept for the caller.  kChains = 2 halves the dependent FMA chain (the
// spring walk is one long dependency chain), 1 saves the packed add that joins the chains (the repulsion
// pass has enough independent interactions in flight and is bound by the FMA pipe).
template <int H, int kChains = 2>
TL_D float dist2(const float2 (&np)[H], const float2 (&q)[H], float2 (&dl)[H]) {
#pragma unroll
  for (int k = 0; k < H; ++k) dl[k] = __fadd2_rn(q[k], np[k]);
  float2 s0 = __fmul2_rn(dl[0], dl[0]);
  if constexpr (kChains == 1 || H == 1) {
#pragma unroll
    for (int k = 1; k < H; ++k) s0 = __ffma2_rn(dl[k], dl[k], s0);
  } else {
    float2 s1 = __fmul2_rn(dl[1], dl[1]);
#pragma unroll
    for (int k = 2; k < H; ++k) {
      if (k & 1) s1 = __ffma2_rn(dl[k], dl[k], s1);
      else s0 = __ffma2_rn(dl[k], dl[k], s0);
    }
    s0 = __fadd2_rn(s0, s1);
  }
  return s0.x + s0.y;
}

TL_D float lg2_approx(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
TL_D float ex2_approx(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// One-sided repulsion of partner q on the point -np: acc += (q - p) / (|q - p| + 0.01)^3.
// The cube and its reciprocal as 2^(-3 log2(ds)) on the special-function unit (two MUFU + one multiply) instead of two
// multiplies + MUFU.RCP: one FMA-pipe slot less in a loop that is bound by that pipe.
template <int H>
TL_D void repel(const float2 (&np)[H], const float2 (&q)[H], float2 (&acc)[H]) {
  float2 dl[H];
  const float d2 = dist2<H, 1>(np, q, dl);
  const float ds = sqrt_approx(d2) + 0.01f;
  const float w = ex2_approx(-3.0f * lg2_approx(ds));
  const float2 ww = make_float2(w, w);
#pragma unroll
  for (int k = 0; k < H; ++k) acc[k] = __ffma2_rn(dl[k], ww, acc[k]);
}

// Every thread of the CTA calls this; returns false when the peers did not arrive in time (the fit is
// then stopped with an error instead of hanging the device).
TL_D bool wait_epoch(const RowDev& dv, unsigned epoch) {
  if (dv.G <= 1 || epoch == 0 || dv.no_wait) return true;
  __shared__ int ok_s;
  if (threadIdx.x < 32) {
    const unsigned* f = dv.flags[dv.rank] + (size_t)(threadIdx.x < (unsigned)dv.G ? threadIdx.x : dv.rank) * kFlagStride;
    const unsigned long long t0 = global_ns();
    bool ok = true;
    for (;;) {
      const unsigned v = ld_acquire_sys(f);
      if (__all_sync(0xffffffffu, v >= epoch)) break;
      if (global_ns() - t0 > kWaitNs) { ok = false; break; }
      __nanosleep(200);
    }
    ok = __all_sync(0xffffffffu, ok);
    if (threadIdx.x == 0) ok_s = ok ? 1 : 0;
  }
  __syncthreads();
  const bool ok = ok_s != 0;
  __syncthreads();
  return ok;
}
TL_D void peer_timeout(const RowDev& dv) {   // one thread
  dv.state->status = 3; dv.state->stop = 1;
  if (dv.host_flag) { __threadfence_system(); dv.host_flag[0] = 1; }
}
// One thread, after a __threadfence_system() that covers the data: tell every replica that this rank reached `epoch`.
TL_D void signal_epoch(const RowDev& dv, unsigned epoch) {
  for (int q = 0; q < dv.G; ++q) st_release_sys(dv.flags[q] + (size_t)dv.rank * kFlagStride, epoch);
}
// All threads call; true in every thread of the CTA that finished last.
TL_D bool last_cta(unsigned* counter) {
  __shared__ int last_s;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(counter, 1u);
    last_s = (t == gridDim.x - 1) ? 1 : 0;
    if (last_s) { *counter = 0u; __threadfence_system(); }
  }
  __syncthreads();
  return last_s != 0;
}

// ---------------------------------------------------------------------------------------------------
// repulsion: one work item = 256 own rows (R per thread) x one chunk of <= 2048 partners
// ---------------------------------------------------------------------------------------------------
// Items are handed out by an atomic counter (reset by combine_kernel's last CTA): the partial sums of an
// item do not depend on which CTA computed it, so the result is the same whatever the residency pattern.
template <int H, int R, int U, int MAXR>
__global__ void __maxnreg__(MAXR) repulse_kernel(RowDev dv, int cur, unsigned epoch) {
  extern __shared__ float4 smem4[];
  __shared__ long long item_s;
  float* sm = reinterpret_cast<float*>(smem4);
  constexpr int T = kRowTile / R;
  constexpr int Dp = Row<H>::kStride;
  constexpr int kStageFloats = kStageJ * Dp;
  if (__ldcg(&dv.state->stop)) return;
  if (dv.adaptive && form_is_tensor(dv)) return;
  if (!wait_epoch(dv, epoch)) { if (blockIdx.x == 0 && threadIdx.x == 0) peer_timeout(dv); return; }
  const int tid = threadIdx.x;
  const float* __restrict__ P = dv.pos[dv.rank] + (size_t)cur * dv.cap_rows * Dp;
  const int tiles = dv.rows / kRowTile;
  const long long items = (long long)tiles * dv.chunks;
  for (;;) {
    if (tid == 0) item_s = (long long)atomicAdd(&dv.counters[2], 1u);
    __syncthreads();
    const long long item = item_s;
    if (item >= items) break;
    const int c = (int)(item / tiles), tile = (int)(item % tiles);
    const int lrow0 = tile * kRowTile;
    float2 np[R][H], acc[R][H];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float2 p[H];
      ld_point<H>(P + (size_t)(dv.row0 + lrow0 + tid + r * T) * Dp, p);
#pragma unroll
      for (int k = 0; k < H; ++k) { np[r][k] = make_float2(-p[k].x, -p[k].y); acc[r][k] = make_float2(0.f, 0.f); }
    }
    const int j0 = c * kChunk;
    const int cnt = min(kChunk, dv.n - j0);
    const int nst = (cnt + kStageJ - 1) / kStageJ;
    const float* __restrict__ src = P + (size_t)j0 * Dp;
    auto prefetch = [&](int s) {
      if (s < nst) {
        const float4* g = reinterpret_cast<const float4*>(src + (size_t)s * kStageFloats);
        float4* d = reinterpret_cast<float4*>(sm + (size_t)(s % kStages) * kStageFloats);
        for (int x = tid; x < kStageFloats / 4; x += T) cp_async16(d + x, g + x);
      }
      cp_async_commit();
    };
#pragma unroll
    for (int s = 0; s < kStages - 1; ++s) prefetch(s);
    for (int s = 0; s < nst; ++s) {
      cp_async_wait<kStages - 2>();
      __syncthreads();
      prefetch(s + kStages - 1);
      const float* __restrict__ q_s = sm + (size_t)(s % kStages) * kStageFloats;
      const int m = min(kStageJ, cnt - s * kStageJ);
#pragma unroll U
      for (int j = 0; j < m; ++j) {
        float2 q[H];
        ld_point<H>(q_s + j * Dp, q);
#pragma unroll
        for (int r = 0; r < R; ++r) repel<H>(np[r], q, acc[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
      st_point<H>(dv.rpart + ((size_t)c * dv.rows + lrow0 + tid + r * T) * Dp, acc[r]);
    __syncthreads();   // the stages are refilled by the next item's prologue; item_s is rewritten
  }
}

#include "rowblock_tc2.cuh"

// ---------------------------------------------------------------------------------------------------
// the walk over the records of the own rows (springs and edge MAE)
// ---------------------------------------------------------------------------------------------------
// One thread per row, one warp per slice of 32 rows; step s of a warp handles record at(s) of each of its 32
// rows.  The partner rows are gathered into a per-warp shared-memory ring kRing steps ahead by cp.async, the
// four lanes of a quad fetching the 16-byte pieces of each other's rows: a warp-wide gather instruction then
// touches 8 cache lines instead of 32 (scattered 16-byte loads are bound by the L1 tag stage, one line per clock,
// long before L2 bandwidth), nothing is held in registers while in flight, and the records themselves ride the
// same ring (8 bytes per lane, one contiguous 256-byte line per warp and step).
constexpr int kRecAhead = 32;   // steps the record stream is prefetched into L2 ahead of its use
constexpr unsigned kSlotMask = 0x3fffffffu;

// kRing = steps of partner rows in flight per warp: 4 when the chip is full of warps (throughput: more CTAs per
// SM), 8 when a rank owns few rows (latency: a step then costs its dependent arithmetic, not an L2 round trip / 3).
template <int H, int kRing>
struct Ring {
  static constexpr int kRecRing = 2 * kRing;
  static constexpr int Dp = Row<H>::kStride;
  static constexpr int NC = Dp / 4;                         // 16-byte pieces of a row
  static constexpr int kRowBytes = NC > 4 ? 128 : NC * 16;  // rows of 5..8 pieces (ndim 17..32) take 128 bytes
  static constexpr int kSlotBytes = 32 * kRowBytes;
  static constexpr int kWarpBytes = kRing * kSlotBytes + kRecRing * 32 * 8;
  // piece c of the row staged for `lane`.  Rows are stored lane-transposed ((lane & 3) * 8 + lane / 4): the 32
  // copies of one gather instruction (fixed quad member u, all quads, all pieces) then fill one contiguous
  // 8-row block - no bank conflict on the write side (the natural order gave 8-way conflicts: the L1 data pipe
  // was the limiter of the walk) - and 64-byte rows rotate their pieces by lane & 3 so that the eight lanes of a
  // 128-bit read phase hit eight different bank groups.  128-byte rows rotate by lane & 7 for the same reason; on the
  // write side the two quads of a phase (lane & 7 = 4 (quad & 1) + u) then cover pieces c ^ u and c ^ u ^ 4: again eight groups.
  static TL_D int piece(int lane, int c) {
    const int row = (lane & 3) * 8 + (lane >> 2);
    if constexpr (NC > 4) return row * 128 + ((c ^ (lane & 7)) << 4);
    return NC == 4 ? row * 64 + ((c ^ (lane & 3)) << 4) : row * kRowBytes + (c << 4);
  }
};

TL_D void cp_async16_ca(unsigned smem_addr, const void* gmem) {
  // through L1: the two 16-byte halves of a 32-byte sector are asked for by two lanes of the same instruction;
  // the L1-bypassing form (.cg) fetches the sector once per lane (measured: twice the L2 traffic)
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gmem) : "memory");
}

TL_D void keep(unsigned& x) { asm volatile("" : "+r"(x)); }   // opaque to the compiler: computed once, not rematerialised in the loop
TL_D uint4 lds128(unsigned a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v; }
TL_D uint2 lds64(unsigned a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }

// consume(record, partner row) is called for every step in order, by all lanes of the warp together.
// Order inside a step (a lone warp per scheduler issues in order, so the order is the schedule): wait for the
// step's data, read it (row pieces, own record, the four records of the quad for the gather) in one burst of
// shared-memory loads, issue the gathers of step t + kRing - 1 and the record of step t + 2 kRing - 1, then the
// arithmetic of step t, which the compiler is free to spread between the copy instructions.
template <int H, int kRing, class F>
TL_D void walk_rows(const float* __restrict__ P, const uint2* __restrict__ rec /* + lane */, int width, int start, char* wsm,
                    F&& consume) {
  typedef Ring<H, kRing> R;
  constexpr int kRecRing = R::kRecRing;
  constexpr unsigned kRowsBytes = kRing * R::kSlotBytes, kRecSlotBytes = 32 * 8;
  const int lane = threadIdx.x & 31;
  const unsigned rows_a = (unsigned)__cvta_generic_to_shared(wsm);
  const unsigned recs_a = rows_a + kRowsBytes;
  const int c = lane & 3, quad = lane & ~3;
  // lane constants (byte offsets inside a ring slot)
  unsigned dst_off[4], own_off[R::NC];
#pragma unroll
  for (int u = 0; u < 4; ++u) { dst_off[u] = (unsigned)R::piece(quad + u, c); keep(dst_off[u]); }
#pragma unroll
  for (int k = 0; k < R::NC; ++k) { own_off[k] = (unsigned)R::piece(lane, k); keep(own_off[k]); }
  unsigned rec_own = (unsigned)lane * 8u, rec_quad = (unsigned)quad * 8u;
  keep(rec_own); keep(rec_quad);
  const char* P_c = reinterpret_cast<const char*>(P) + c * 16;
  asm volatile("" : "+l"(P_c));
  asm volatile("" : "+l"(rec));
  // cursors (warp-uniform)
  int r_at = start, r_left = width;
  unsigned r_slot_a = recs_a;                                  // record-ring slot the next record goes to
  int pf_at = start + kRecAhead;                               // record line pulled into L2 this step (lanes 0, 1)
  if (width > 0) pf_at %= width;
  const uint2* rec_line = rec - lane + (lane & 1) * 16;
  auto issue_rec = [&]() {
    if (r_left > 0) {
      if (lane < 2 && r_left > kRecAhead) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec_line + (size_t)pf_at * 32));
      pf_at = (pf_at + 1 == width) ? 0 : pf_at + 1;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(r_slot_a + rec_own), "l"(rec + (size_t)r_at * 32) : "memory");
      r_at = (r_at + 1 == width) ? 0 : r_at + 1;
      --r_left;
    }
    r_slot_a = (r_slot_a + kRecSlotBytes == recs_a + kRecRing * kRecSlotBytes) ? recs_a : r_slot_a + kRecSlotBytes;
  };
  int g_left = width;
  unsigned g_slot_a = rows_a, g_rslot_a = recs_a;               // row-ring slot gathered into, record slot it reads
  auto issue_gather = [&](const uint4 ja, const uint4 jb) {     // the four records of the quad: (ja.x, ja.z, jb.x, jb.z) are the .x words
    if (g_left > 0) {
      if (c < R::NC) {
        const unsigned j[4] = {ja.x & kSlotMask, ja.z & kSlotMask, jb.x & kSlotMask, jb.z & kSlotMask};
#pragma unroll
        for (int u = 0; u < 4; ++u) cp_async16_ca(g_slot_a + dst_off[u], P_c + (size_t)j[u] * (R::Dp * 4));
        if constexpr (R::NC > 4) {                  // rows of more than four pieces: this lane also fetches piece c + 4
          if (c + 4 < R::NC) {                      // piece(l, c + 4) = piece(l, c) ^ 64 (c < 4: (c + 4) ^ f = (c ^ f) ^ 4)
#pragma unroll
            for (int u = 0; u < 4; ++u) cp_async16_ca(g_slot_a + (dst_off[u] ^ 64u), P_c + (size_t)j[u] * (R::Dp * 4) + 64);
          }
        }
      }
      --g_left;
    }
    g_slot_a = (g_slot_a + R::kSlotBytes == rows_a + kRowsBytes) ? rows_a : g_slot_a + R::kSlotBytes;
    g_rslot_a = (g_rslot_a + kRecSlotBytes == recs_a + kRecRing * kRecSlotBytes) ? recs_a : g_rslot_a + kRecSlotBytes;
  };
  for (int st = 0; st < kRecRing - 1; ++st) issue_rec();
  cp_async_commit();
  cp_async_wait<0>();
  __syncwarp();
  for (int st = 0; st < kRing - 1; ++st) {
    const uint4 ja = lds128(g_rslot_a + rec_quad), jb = lds128(g_rslot_a + rec_quad + 16);
    issue_gather(ja, jb);
    cp_async_commit();
  }
  unsigned slot_a = rows_a, rslot_a = recs_a;
  for (int t = 0; t < width; ++t) {
    cp_async_wait<kRing - 2>();
    __syncwarp();
    // ---- everything this step reads from shared memory ----
    uint4 qv[R::NC];
#pragma unroll
    for (int k = 0; k < H / 2; ++k) {
      // 128-byte rows: piece(lane, k) = piece(lane, 0) ^ (k << 4); one register instead of eight
      if constexpr (R::NC > 4) qv[k] = lds128(slot_a + (own_off[0] ^ ((unsigned)k << 4)));
      else qv[k] = lds128(slot_a + own_off[k]);
    }
    uint2 qt = make_uint2(0u, 0u);
    if constexpr (H % 2 == 1) qt = lds64(slot_a + own_off[H / 2]);
    const uint2 r = lds64(rslot_a + rec_own);
    const uint4 ja = lds128(g_rslot_a + rec_quad), jb = lds128(g_rslot_a + rec_quad + 16);
    // ---- copies for the steps ahead ----
    issue_gather(ja, jb);
    issue_rec();
    cp_async_commit();
    slot_a = (slot_a + R::kSlotBytes == rows_a + kRowsBytes) ? rows_a : slot_a + R::kSlotBytes;
    rslot_a = (rslot_a + kRecSlotBytes == recs_a + kRecRing * kRecSlotBytes) ? recs_a : rslot_a + kRecSlotBytes;
    // ---- this step ----
    float2 q[H];
#pragma unroll
    for (int k = 0; k < H / 2; ++k) {
      q[2 * k] = make_float2(__uint_as_float(qv[k].x), __uint_as_float(qv[k].y));
      q[2 * k + 1] = make_float2(__uint_as_float(qv[k].z), __uint_as_float(qv[k].w));
    }
    if constexpr (H % 2 == 1) q[H - 1] = make_float2(__uint_as_float(qt.x), __uint_as_float(qt.y));
    consume(r, q);
  }
  cp_async_wait<0>();
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------
// springs: one thread per own row, Gauss-Seidel along the row
// ---------------------------------------------------------------------------------------------------
// Launched with kBlockRows threads; a CTA walks row blocks blockIdx.x, + gridDim.x, ...  112 registers: 128 x 112 =
// 14,336, what two CTAs of repulse_tc2_kernel (320 x 80) leave of the SM's 65,536, so one walk CTA per SM runs beside
// them (launch_iteration; tests/test_resource_budget.py).
template <int H, int kRing>
__global__ void __maxnreg__(H <= 8 ? kWalkRegs : kWalkRegsWide) spring_kernel(RowDev dv, FitParams prm, int cur, unsigned epoch) {
  constexpr int Dp = Row<H>::kStride;
  extern __shared__ float4 smem4[];
  asm volatile("griddepcontrol.launch_dependents;");   // a repulsion pass launched as programmatic dependent may start now
  if (__ldcg(&dv.state->stop)) return;
  if (!wait_epoch(dv, epoch)) { if (blockIdx.x == 0 && threadIdx.x == 0) peer_timeout(dv); return; }
  const int tid = threadIdx.x;
  const float* __restrict__ P = dv.pos[dv.rank] + (size_t)cur * dv.cap_rows * Dp;
  const float k = (float)__ldcg(&dv.state->k);
  const int iter = __ldcg(&dv.state->iter);
  for (int blk = blockIdx.x; blk < dv.rows / kBlockRows; blk += gridDim.x) {
  const int lrow = blk * kBlockRows + tid;                 // row inside the own block
  const int row = dv.row0 + lrow;                          // slot
  const float dp1 = dv.dp1[row];                           // 0 for a padding row: its lane walks along, stores nothing
  const float safe = dp1 > 0.f ? dp1 : 1.f;
  float2 p0n[H], xn[H];   // -P_i and -x (the running position, negated: deltas are q + (-x))
  {
    float2 p[H];
    ld_point<H>(P + (size_t)row * Dp, p);
#pragma unroll
    for (int kk = 0; kk < H; ++kk) { p0n[kk] = make_float2(-p[kk].x, -p[kk].y); xn[kk] = p0n[kk]; }
  }
  const float rdeg = (float)(0.5 * prm.c_repulsion) / safe;
  const float two_k_rnorm = 2.0f * k / (4.0f * safe + k);
  const int slice = lrow >> 5;
  const int width = dv.swidth[slice];
  int start = 0;
  if (width > 0) start = (int)(mix64(dv.seed ^ mix64(((unsigned long long)(unsigned)iter << 32) | (unsigned)(row >> 5))) % (unsigned long long)width);
  walk_rows<H, kRing>(P, dv.recs + dv.soff[slice] + (tid & 31), width, start,
               reinterpret_cast<char*>(smem4) + (size_t)(tid >> 5) * Ring<H, kRing>::kWarpBytes, [&](const uint2 r, const float2 (&q)[H]) {
    const unsigned type = r.x >> 30;
    const float target = __uint_as_float(r.y);
    float2 dl[H], d0[H];
    const float d2 = dist2<H>(xn, q, dl);
    const float e2 = dist2<H>(p0n, q, d0);
    const float dist = sqrt_approx(d2);
    const bool spring = type == 0u || (type == 1u ? dist < target : (type == 2u && dist > target));   // :237-243
    const float ds0 = sqrt_approx(e2) + 0.01f;
    const float w0 = spring ? rdeg * rcp_approx(ds0 * ds0 * ds0) : 0.f;
    const float f = spring ? two_k_rnorm * (target - dist) * rcp_approx(dist + 0.01f) : 0.f;
    // x += -delta f + d0 w0  <=>  (-x) += delta f - d0 w0; the take-back term does not wait for f
    const float2 ff = make_float2(f, f), nw = make_float2(-w0, -w0);
    if constexpr (H <= 8) {
#pragma unroll
      for (int kk = 0; kk < H; ++kk) xn[kk] = __ffma2_rn(dl[kk], ff, __ffma2_rn(d0[kk], nw, xn[kk]));
    } else {
      // ndim 17..32: both delta arrays held across the weights do not fit beside the rows (spills); they are recomputed
      // from q, the same roundings.  q is passed through an empty asm so that the compiler cannot merge the two sums
      // back into the ones of dist2 and keep dl / d0 alive after all.
      float2 qr[H];
#pragma unroll
      for (int kk = 0; kk < H; ++kk) { qr[kk] = q[kk]; asm volatile("" : "+f"(qr[kk].x), "+f"(qr[kk].y)); }
#pragma unroll
      for (int kk = 0; kk < H; ++kk)
        xn[kk] = __ffma2_rn(__fadd2_rn(qr[kk], xn[kk]), ff, __ffma2_rn(__fadd2_rn(qr[kk], p0n[kk]), nw, xn[kk]));
    }
  });
  if (dp1 > 0.f) {
    float2 x[H];
#pragma unroll
    for (int kk = 0; kk < H; ++kk) x[kk] = make_float2(-xn[kk].x, -xn[kk].y);
    st_point<H>(dv.xs + (size_t)lrow * Dp, x);
  }
  }
}

// ---------------------------------------------------------------------------------------------------
// combine: P'_i = (position after the springs) + (repulsion of the iteration), stored into every replica
// ---------------------------------------------------------------------------------------------------
// The spring walk (a long dependent chain per row: latency) and the repulsion pass (issue and special-function
// throughput) both read only the iteration's snapshot, so they run side by side (the walk is a programmatic dependent
// launch of the pass: it starts as soon as the pass's CTAs are resident); this kernel, a normal launch after both,
// waits for both grids and joins them.  The repulsion sums of a row are added chunk by chunk in a fixed order (the
// result does not depend on the rank count).
template <int H>
__global__ void __launch_bounds__(kBlockRows) combine_kernel(RowDev dv, FitParams prm, int cur, unsigned epoch) {
  constexpr int Dp = Row<H>::kStride;
  if (__ldcg(&dv.state->stop)) return;
  const int tid = threadIdx.x;
  const int lrow = blockIdx.x * kBlockRows + tid;
  const int row = dv.row0 + lrow;
  const float dp1 = dv.dp1[row];
  if (dp1 > 0.f) {
    float2 x[H], rs[H];
    ld_point<H>(dv.xs + (size_t)lrow * Dp, x);
#pragma unroll
    for (int kk = 0; kk < H; ++kk) rs[kk] = make_float2(0.f, 0.f);
    const int nparts = (dv.adaptive && !form_is_tensor(dv)) ? dv.chunks : dv.rparts;   // the FP32 form writes one entry per chunk
    for (int c = 0; c < nparts; ++c) {
      float2 t[H];
      ld_point<H>(dv.rpart + ((size_t)c * dv.rows + lrow) * Dp, t);
#pragma unroll
      for (int kk = 0; kk < H; ++kk) rs[kk] = __fadd2_rn(rs[kk], t[kk]);
    }
    const float nrdeg = -(float)(0.5 * prm.c_repulsion) / dp1;     // R_i = -sum * (c / 2) / (deg_i + 1)
    const float2 rr = make_float2(nrdeg, nrdeg);
#pragma unroll
    for (int kk = 0; kk < H; ++kk) x[kk] = __ffma2_rn(rs[kk], rr, x[kk]);
    const size_t o = ((size_t)(cur ^ 1) * dv.cap_rows + row) * Dp;
    for (int g = 0; g < dv.G; ++g) st_point<H>(dv.pos[g] + o, x);   // own replica and every peer (NVLink stores)
  }
  if (last_cta(&dv.counters[0])) {
    if (tid == 0) {
      FitState* st = dv.state;
      const int iter = st->iter;
      st->k = st->k * (1.0 - prm.cooling_rate);         // :289
      st->iter = iter + 1;
      st->pair_updates += dv.pairs_per_iter;
      dv.counters[2] = 0u;                              // the repulsion pass of the next iteration starts at item 0
      if (dv.host_flag) dv.host_flag[1] = iter + 1;
      __threadfence_system();
      signal_epoch(dv, epoch);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// edge MAE on the new positions: one thread per own row over the records this rank counts
// ---------------------------------------------------------------------------------------------------
template <int H, int kRing>
__global__ void __launch_bounds__(kBlockRows) mae_kernel(RowDev dv, int nxt, unsigned wait_for, unsigned epoch) {
  constexpr int Dp = Row<H>::kStride;
  extern __shared__ float4 smem4[];
  __shared__ double red_s[3][kBlockRows / 32];
  if (__ldcg(&dv.state->stop)) return;
  if (!wait_epoch(dv, wait_for)) { if (blockIdx.x == 0 && threadIdx.x == 0) peer_timeout(dv); return; }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lrow = blockIdx.x * kBlockRows + tid;
  const int row = dv.row0 + lrow;
  const float* __restrict__ P = dv.pos[dv.rank] + (size_t)nxt * dv.cap_rows * Dp;
  double sum = 0.0, cnt = 0.0, bad = 0.0;
  float2 pn[H];
  {
    float2 p[H];
    ld_point<H>(P + (size_t)row * Dp, p);
#pragma unroll
    for (int kk = 0; kk < H; ++kk) {
      if (!isfinite(p[kk].x) || !isfinite(p[kk].y)) bad = 1.0;
      pn[kk] = make_float2(-p[kk].x, -p[kk].y);
    }
  }
  const int slice = lrow >> 5;
  walk_rows<H, kRing>(P, dv.mrecs + dv.moff[slice] + lane, dv.mwidth[slice], 0,
               reinterpret_cast<char*>(smem4) + (size_t)warp * Ring<H, kRing>::kWarpBytes, [&](const uint2 r, const float2 (&q)[H]) {
    float2 dl[H];
    const float dist = __fsqrt_rn(dist2<H>(pn, q, dl));
    const unsigned type = r.x >> 30;
    const float target = __uint_as_float(r.y);
    const bool on = type == 0u || (type == 1u ? dist < target : (type == 2u && dist > target));   // :72-75
    if (on) { sum += fabs((double)target - (double)dist); cnt += 1.0; }
  });
  // fixed tree: lanes, then warps
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_down_sync(0xffffffffu, sum, o);
    cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    bad += __shfl_down_sync(0xffffffffu, bad, o);
  }
  if (lane == 0) { red_s[0][warp] = sum; red_s[1][warp] = cnt; red_s[2][warp] = bad; }
  __syncthreads();
  if (tid == 0) {
    double s = 0.0, c = 0.0, b = 0.0;
    for (int w = 0; w < kBlockRows / 32; ++w) { s += red_s[0][w]; c += red_s[1][w]; b += red_s[2][w]; }
    const size_t e = (size_t)(row / kBlockRows) * 4;
    for (int g = 0; g < dv.G; ++g) {
      double* o = dv.red[g] + e;
      o[0] = s; o[1] = c; o[2] = b;
    }
  }
  if (last_cta(&dv.counters[1]) && tid == 0) signal_epoch(dv, epoch);
}

// ---------------------------------------------------------------------------------------------------
// controller (one CTA): pooled MAE, three-way classification, finite check
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ctl_kernel(RowDev dv, FitParams prm, int check, int fin, unsigned wait_for) {
  __shared__ double red_s[3][256];
  if (__ldcg(&dv.state->stop)) return;
  if (!wait_epoch(dv, wait_for)) { if (threadIdx.x == 0) peer_timeout(dv); return; }
  const int tid = threadIdx.x;
  const int entries = dv.slots / kBlockRows;
  const double* __restrict__ red = dv.red[dv.rank];
  double s = 0.0, c = 0.0, b = 0.0;
  for (int e = tid; e < entries; e += 256) { s += __ldcg(red + (size_t)e * 4); c += __ldcg(red + (size_t)e * 4 + 1); b += __ldcg(red + (size_t)e * 4 + 2); }
  red_s[0][tid] = s; red_s[1][tid] = c; red_s[2][tid] = b;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) { red_s[0][tid] += red_s[0][tid + o]; red_s[1][tid] += red_s[1][tid + o]; red_s[2][tid] += red_s[2][tid + o]; }
    __syncthreads();
  }
  if (tid == 0) {
    FitState st = *dv.state;
    const int iter = st.iter - 1;   // the iteration that just finished
    st.snapshot = 0;
    if (check) {
      controller_check(st, prm, iter, red_s[0][0], (long long)red_s[1][0]);
      if (dv.trace && iter >= 0 && iter < prm.n_iter) dv.trace[iter] = st.last_error;
    }
    if (!st.stop && fin && red_s[2][0] > 0.0) { st.status = 2; st.fail_iter = iter + 1; st.stop = 1; }
    *dv.state = st;
    if (dv.host_flag && st.stop) { __threadfence_system(); dv.host_flag[0] = 1; }
  }
}

__global__ void __launch_bounds__(256) snap_kernel(RowDev dv, int nxt) {
  if (!__ldcg(&dv.state->snapshot)) return;
  const size_t total4 = (size_t)dv.slots * dv.Dp / 4;
  const float4* __restrict__ src = reinterpret_cast<const float4*>(dv.pos[dv.rank] + (size_t)nxt * dv.cap_rows * dv.Dp);
  float4* dst = reinterpret_cast<float4*>(dv.best);
  for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < total4; x += (size_t)gridDim.x * blockDim.x) dst[x] = src[x];
}

// ---------------------------------------------------------------------------------------------------
// set-up kernels: COO edge list -> the two SELL-32 record arrays of the own rows
// ---------------------------------------------------------------------------------------------------
// A pair is counted in the MAE by exactly one of its endpoints, the two halves of every row about equal.
TL_HD bool counts_here(uint32_t self, uint32_t other) { return (((self + other) & 1u) != 0u) == (self < other); }

__global__ void count_kernel(const int32_t* __restrict__ ei, const int32_t* __restrict__ ej, long long E, long long n,
                             const int32_t* __restrict__ slot_of_point, int row0, int rows, unsigned* len, unsigned* mlen, int* bad) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    const long long a = ei[e], b = ej[e];
    if (a < 0 || b < 0 || a >= n || b >= n || a == b) { *bad = 1; continue; }
    const uint32_t sa = (uint32_t)slot_of_point[a], sb = (uint32_t)slot_of_point[b];
    const int la = (int)sa - row0, lb = (int)sb - row0;
    if (la >= 0 && la < rows) { atomicAdd(&len[la], 1u); if (counts_here(sa, sb)) atomicAdd(&mlen[la], 1u); }
    if (lb >= 0 && lb < rows) { atomicAdd(&len[lb], 1u); if (counts_here(sb, sa)) atomicAdd(&mlen[lb], 1u); }
  }
}
__global__ void fill_kernel(const int32_t* __restrict__ ei, const int32_t* __restrict__ ej, const double* __restrict__ dist,
                            const int32_t* __restrict__ thr, long long E, const int32_t* __restrict__ slot_of_point, int row0,
                            int rows, const unsigned long long* __restrict__ off, unsigned* cursor, uint2* tmp) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    const uint32_t sa = (uint32_t)slot_of_point[ei[e]], sb = (uint32_t)slot_of_point[ej[e]];
    const int t = thr[e];
    const unsigned type = t == 0 ? 0u : (t == 1 ? 1u : 2u);   // src/optimization.cpp:237-243
    const unsigned tb = __float_as_uint((float)dist[e]);
    const int la = (int)sa - row0, lb = (int)sb - row0;
    if (la >= 0 && la < rows) tmp[off[la] + atomicAdd(&cursor[la], 1u)] = make_uint2(sb | (type << 30), tb);
    if (lb >= 0 && lb < rows) tmp[off[lb] + atomicAdd(&cursor[lb], 1u)] = make_uint2(sa | (type << 30), tb);
  }
}
// One warp per own row: sort the row's records by (partner, type, target bits) - a fixed order whatever the
// scatter left - and write them, transposed, into the slices; the tail of a row up to the slice width is
// padding (type 3: never a spring, never counted; partner = the row itself).  Rows of up to kSortCap records
// are sorted in shared memory (bitonic network on the 64-bit keys, from which the record is rebuilt), longer
// ones by counting ranks in global memory.
constexpr int kSortCap = 2048;
TL_D unsigned long long rec_key(uint2 r) {
  return ((unsigned long long)(r.x & 0x3fffffffu) << 34) | ((unsigned long long)(r.x >> 30) << 32) | r.y;
}
TL_D uint2 key_rec(unsigned long long k) {
  return make_uint2((unsigned)(k >> 34) | ((unsigned)((k >> 32) & 3ull) << 30), (unsigned)k);
}
__global__ void __launch_bounds__(128) sell_kernel(const uint2* __restrict__ tmp, const unsigned long long* __restrict__ off,
                                                   const unsigned* __restrict__ len, int row0, int rows,
                                                   const unsigned long long* __restrict__ soff, const int* __restrict__ swidth,
                                                   const unsigned long long* __restrict__ moff, const int* __restrict__ mwidth,
                                                   uint2* recs, uint2* mrecs) {
  extern __shared__ unsigned long long sort_s[];   // [4][kSortCap]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lrow = blockIdx.x * 4 + warp;
  if (lrow >= rows) return;
  const unsigned n = len[lrow];
  const uint2* __restrict__ in = tmp + off[lrow];
  const uint32_t self = (uint32_t)(row0 + lrow);
  const int slice = lrow >> 5, rl = lrow & 31;
  uint2* out = recs + soff[slice] + rl;
  uint2* mout = mrecs + moff[slice] + rl;
  unsigned mcount = 0;
  if (n <= (unsigned)kSortCap) {
    unsigned long long* ks = sort_s + (size_t)warp * kSortCap;
    unsigned m = 32;
    while (m < n) m <<= 1;
    for (unsigned x = lane; x < m; x += 32) ks[x] = x < n ? rec_key(in[x]) : ~0ull;
    __syncwarp();
    for (unsigned k = 2; k <= m; k <<= 1)
      for (unsigned j = k >> 1; j > 0; j >>= 1) {
        for (unsigned i = lane; i < m; i += 32) {
          const unsigned l = i ^ j;
          if (l > i) {
            const unsigned long long a = ks[i], b = ks[l];
            if ((a > b) == ((i & k) == 0)) { ks[i] = b; ks[l] = a; }
          }
        }
        __syncwarp();
      }
    for (unsigned x0 = 0; x0 < n; x0 += 32) {
      const unsigned x = x0 + lane;
      const uint2 r = x < n ? key_rec(ks[x]) : make_uint2(0u, 0u);
      const bool counted = x < n && counts_here(self, r.x & 0x3fffffffu);
      const unsigned vote = __ballot_sync(0xffffffffu, counted);
      if (x < n) out[(size_t)x * 32] = r;
      if (counted) mout[(size_t)(mcount + __popc(vote & ((1u << lane) - 1u))) * 32] = r;
      mcount += __popc(vote);
    }
  } else {
    for (unsigned x0 = 0; x0 < n; x0 += 32) {
      const unsigned x = x0 + lane;
      if (x < n) {
        const uint2 r = in[x];
        const unsigned long long mkey = rec_key(r);
        const bool mcounted = counts_here(self, r.x & 0x3fffffffu);
        unsigned rank = 0, mrank = 0;
        for (unsigned y = 0; y < n; ++y) {
          const uint2 o = in[y];
          const unsigned long long okey = rec_key(o);
          const bool before = okey < mkey || (okey == mkey && y < x);
          rank += before ? 1u : 0u;
          mrank += (before && counts_here(self, o.x & 0x3fffffffu)) ? 1u : 0u;
        }
        out[(size_t)rank * 32] = r;
        if (mcounted) mout[(size_t)mrank * 32] = r;
      }
    }
    for (unsigned y = lane; y < n; y += 32) mcount += counts_here(self, in[y].x & 0x3fffffffu) ? 1u : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mcount += __shfl_xor_sync(0xffffffffu, mcount, o);
  }
  const uint2 pad = make_uint2(self | (3u << 30), 0u);
  for (unsigned x = n + lane; x < (unsigned)swidth[slice]; x += 32) out[(size_t)x * 32] = pad;
  for (unsigned x = mcount + lane; x < (unsigned)mwidth[slice]; x += 32) mout[(size_t)x * 32] = pad;
}

template <class F>
void dispatch_h(int H, F&& f) {
  switch (H) {
    case 1: f(std::integral_constant<int, 1>()); break;
    case 2: f(std::integral_constant<int, 2>()); break;
    case 3: f(std::integral_constant<int, 3>()); break;
    case 4: f(std::integral_constant<int, 4>()); break;
    case 5: f(std::integral_constant<int, 5>()); break;
    case 6: f(std::integral_constant<int, 6>()); break;
    case 7: f(std::integral_constant<int, 7>()); break;
    case 8: f(std::integral_constant<int, 8>()); break;
    case 10: f(std::integral_constant<int, 10>()); break;
    case 12: f(std::integral_constant<int, 12>()); break;
    case 14: f(std::integral_constant<int, 14>()); break;
    case 16: f(std::integral_constant<int, 16>()); break;
    default: throw BadArg("row-block mode supports ndim <= 32 (the replay mode takes any ndim)");
  }
}

// Packed coordinate pairs a row is computed on.  ndim 17..32 runs on the whole padded row (Row<H>::kStride = 2 H): the
// pad columns are zero, their deltas and updates stay +-0 and add +0 to every sum, so the real coordinates come out as
// without the pad, and four instantiations cover sixteen ndims.
int row_h(int ndim) { return ndim <= 16 ? (ndim + 1) / 2 : (ndim + 3) / 4 * 2; }

}  // namespace

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
struct RowHandle {            // what a rank publishes: its shared block and the geometry the others must agree with
  cudaIpcMemHandle_t mem;
  int32_t rank, n_ranks, slots, Dp;
  uint64_t layout;            // byte size of the shared block
};

struct RowPlan {
  int device = 0;
  int64_t n = 0, E = 0;
  RowDev dv{};
  FitParams prm{};
  std::vector<int32_t> slot_of_point;
  // shared block (cudaMalloc: exportable): positions [2][cap_rows][Dp] | red [slots/128][4] | flags
  char* shared = nullptr;
  size_t shared_bytes = 0, off_red = 0, off_flags = 0;
  void* peer_base[kMaxShards] = {};   // mapped blocks of the other ranks (IPC) - closed on destroy
  bool peer_ipc[kMaxShards] = {};
  // local
  float* best = nullptr; float* dp1 = nullptr; float* rpart = nullptr; float* xs = nullptr;
  float* tc_buf = nullptr;    // the arrays of T2Image in one allocation
  bool tc_form = false;       // distances and accumulation on the tensor cores (image_tc_kernel, image_t2_kernel, repulse_tc2_kernel)
  int tc_cpi = 1;             // partner chunks per work item
  uint2* recs = nullptr; uint2* mrecs = nullptr;
  unsigned long long* soff = nullptr; unsigned long long* moff = nullptr; int* swidth = nullptr; int* mwidth = nullptr;
  FitState* state = nullptr; double* trace = nullptr; unsigned* counters = nullptr;
  volatile int* h_flag = nullptr; int* d_flag = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int64_t n_holdout = 0;
  std::vector<int32_t> hold_i, hold_j; std::vector<double> hold_truth;
  int iter_launched = 0;      // iterations enqueued so far
  unsigned epoch = 0;         // signals enqueued so far (the same number on every rank)
  int64_t launches = 0;
  int64_t n_recs = 0, n_mrecs = 0;
  int64_t tensor_iters = -1;  // adaptive runs: iterations that ran the tensor form (read back by row_result; -1 = not adaptive / not read yet)
  int rep_ctas = 0;
  int64_t rep_items = 0;      // work items of one pass of the form rep_form names (the tensor form groups tc_cpi chunks per item)
  double near_limit = 0.0;    // adaptive runs: the tensor form while the probed near-pair fraction is at most this
  int rep_form = 0;           // form of the repulsion pass: 11 (two-GEMM tensor-core pass) or 5 (FP32 difference form)
  bool deep_ring = false;
  bool overlap = true;        // repulsion pass launched as programmatic dependent of the spring walk (TOPOLOW_OVERLAP=0: in order)
  int walk_ctas = 0;          // grid of the spring walk under the repulsion pass
  int sm_count = 148;
  void* rep_fn = nullptr;
  int f32_ctas = 0, f32_threads = 128;   // the FP32 difference form beside a tensor form (adaptive runs launch both)
  size_t f32_smem = 0;
  double total_ms = 0.0;
  bool attached = false;

  ~RowPlan() {
    DeviceScope on(device);
    if (stream) cudaStreamSynchronize(stream);
    for (int q = 0; q < kMaxShards; ++q) if (peer_base[q] && peer_ipc[q]) cudaIpcCloseMemHandle(peer_base[q]);
    if (shared) cudaFree(shared);
    pool_free(best); pool_free(dp1); pool_free(rpart); pool_free(xs); pool_free(tc_buf); pool_free(recs); pool_free(mrecs);
    pool_free(soff); pool_free(moff); pool_free(swidth); pool_free(mwidth);
    pool_free(state); pool_free(trace); pool_free(counters);
    if (h_flag) cudaFreeHost((void*)h_flag);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace {

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

void set_self_pointers(RowPlan& rp) {
  RowDev& dv = rp.dv;
  dv.pos[dv.rank] = reinterpret_cast<float*>(rp.shared);
  dv.red[dv.rank] = reinterpret_cast<double*>(rp.shared + rp.off_red);
  dv.flags[dv.rank] = reinterpret_cast<unsigned*>(rp.shared + rp.off_flags);
}
void set_peer_pointers(RowPlan& rp, int q, char* base) {
  rp.dv.pos[q] = reinterpret_cast<float*>(base);
  rp.dv.red[q] = reinterpret_cast<double*>(base + rp.off_red);
  rp.dv.flags[q] = reinterpret_cast<unsigned*>(base + rp.off_flags);
}

// Builds the record arrays of the own rows on the device.
void build_records(RowPlan& rp, const topolow_problem& pb) {
  RowDev& dv = rp.dv;
  cudaStream_t s = rp.stream;
  const long long E = pb.n_edges;
  const int rows = dv.rows, slices = rows / 32;
  AsyncBuf<int32_t> d_ei(E, s), d_ej(E, s), d_thr(E, s), d_slot(rp.slot_of_point.size(), s);
  AsyncBuf<double> d_dist(E, s);
  AsyncBuf<unsigned> d_len(rows, s), d_mlen(rows, s), d_cur(rows, s);
  AsyncBuf<unsigned long long> d_off(rows + 1, s);
  AsyncBuf<int> d_bad(1, s);
  PhaseTimer pt(s);
  TL_CUDA(cudaMemcpyAsync(d_slot, rp.slot_of_point.data(), rp.slot_of_point.size() * 4, cudaMemcpyHostToDevice, s));
  if (E > 0) {
    TL_CUDA(cudaMemcpyAsync(d_ei, pb.edge_i, E * 4, cudaMemcpyHostToDevice, s));
    TL_CUDA(cudaMemcpyAsync(d_ej, pb.edge_j, E * 4, cudaMemcpyHostToDevice, s));
    TL_CUDA(cudaMemcpyAsync(d_dist, pb.edge_dist, E * 8, cudaMemcpyHostToDevice, s));
    TL_CUDA(cudaMemcpyAsync(d_thr, pb.edge_thresh, E * 4, cudaMemcpyHostToDevice, s));
  }
  TL_CUDA(cudaMemsetAsync(d_len, 0, rows * 4, s));
  TL_CUDA(cudaMemsetAsync(d_mlen, 0, rows * 4, s));
  TL_CUDA(cudaMemsetAsync(d_cur, 0, rows * 4, s));
  TL_CUDA(cudaMemsetAsync(d_bad, 0, 4, s));
  pt.mark("rows: host to device");
  const int blocks = 148 * 8, threads = 256;
  if (E > 0) {
    count_kernel<<<blocks, threads, 0, s>>>(d_ei, d_ej, E, pb.n, d_slot, dv.row0, rows, d_len, d_mlen, d_bad);
    TL_CUDA(cudaGetLastError());
  }
  std::vector<unsigned> len(rows), mlen(rows);
  int bad = 0;
  TL_CUDA(cudaMemcpyAsync(len.data(), d_len, rows * 4, cudaMemcpyDeviceToHost, s));
  TL_CUDA(cudaMemcpyAsync(mlen.data(), d_mlen, rows * 4, cudaMemcpyDeviceToHost, s));
  TL_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, s));
  TL_CUDA(cudaStreamSynchronize(s));
  if (bad) throw BadArg("edge index out of range");
  std::vector<unsigned long long> off(rows + 1, 0), soff(slices), moff(slices);
  std::vector<int> swidth(slices), mwidth(slices);
  for (int r = 0; r < rows; ++r) off[r + 1] = off[r] + len[r];
  unsigned long long so = 0, mo = 0;
  for (int sl = 0; sl < slices; ++sl) {
    unsigned w = 0, mw = 0;
    for (int r = 0; r < 32; ++r) { w = std::max(w, len[sl * 32 + r]); mw = std::max(mw, mlen[sl * 32 + r]); }
    soff[sl] = so; moff[sl] = mo; swidth[sl] = (int)w; mwidth[sl] = (int)mw;
    so += (unsigned long long)w * 32; mo += (unsigned long long)mw * 32;
  }
  rp.n_recs = (int64_t)so; rp.n_mrecs = (int64_t)mo;
  pool_alloc(rp.recs, (size_t)so * sizeof(uint2));
  pool_alloc(rp.mrecs, (size_t)mo * sizeof(uint2));
  pool_alloc(rp.soff, slices * sizeof(unsigned long long));
  pool_alloc(rp.moff, slices * sizeof(unsigned long long));
  pool_alloc(rp.swidth, slices * sizeof(int));
  pool_alloc(rp.mwidth, slices * sizeof(int));
  pool_ready();
  AsyncBuf<uint2> d_tmp((size_t)off[rows], s);
  TL_CUDA(cudaMemcpyAsync(d_off, off.data(), (rows + 1) * 8, cudaMemcpyHostToDevice, s));
  TL_CUDA(cudaMemcpyAsync(rp.soff, soff.data(), slices * 8, cudaMemcpyHostToDevice, s));
  TL_CUDA(cudaMemcpyAsync(rp.moff, moff.data(), slices * 8, cudaMemcpyHostToDevice, s));
  TL_CUDA(cudaMemcpyAsync(rp.swidth, swidth.data(), slices * 4, cudaMemcpyHostToDevice, s));
  TL_CUDA(cudaMemcpyAsync(rp.mwidth, mwidth.data(), slices * 4, cudaMemcpyHostToDevice, s));
  pt.mark("rows: lengths + offsets");
  if (E > 0) {
    fill_kernel<<<blocks, threads, 0, s>>>(d_ei, d_ej, d_dist, d_thr, E, d_slot, dv.row0, rows, d_off, d_cur, d_tmp);
    TL_CUDA(cudaGetLastError());
  }
  // per device, so every time (a function-local static would configure only the device of the first call)
  TL_CUDA(cudaFuncSetAttribute(sell_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kSortCap * 8));
  sell_kernel<<<(rows + 3) / 4, 128, 4 * kSortCap * 8, s>>>(d_tmp, d_off, d_len, dv.row0, rows, rp.soff, rp.swidth, rp.moff, rp.mwidth,
                                              rp.recs, rp.mrecs);
  TL_CUDA(cudaGetLastError());
  TL_CUDA(cudaStreamSynchronize(s));   // the host vectors above go out of scope
  pt.mark("rows: fill + sort + transpose");
  dv.recs = rp.recs; dv.mrecs = rp.mrecs; dv.soff = rp.soff; dv.moff = rp.moff; dv.swidth = rp.swidth; dv.mwidth = rp.mwidth;
}

TcImage tc_image(const RowPlan& rp) {
  TcImage im;
  const size_t cap = rp.dv.cap_rows;
  im.xhi = rp.tc_buf; im.xlo = im.xhi + 16 * cap; im.aug_a = im.xlo + 16 * cap; im.aug_b = im.aug_a + 4 * cap; im.rows32 = im.aug_b + 4 * cap;
  return im;
}
T2Image t2_image(const RowPlan& rp) {
  T2Image im;
  im.a = tc_image(rp);
  im.yhi = im.a.rows32 + 16 * rp.dv.cap_rows; im.ylo = im.yhi + 32 * rp.dv.cap_rows;
  return im;
}
template <int H>
void launch_image_tc(RowPlan& rp, cudaStream_t s, int cur, unsigned e_prev) {
  static_assert(H <= 8, "the tensor form takes ndim <= 16");
  image_tc_kernel<H><<<(unsigned)(rp.dv.cap_rows / kBlockRows), kBlockRows, 0, s>>>(rp.dv, tc_image(rp), cur, e_prev);
  image_t2_kernel<<<(unsigned)(rp.dv.cap_rows / 4 * 32 / 256), 256, 0, s>>>(rp.dv, t2_image(rp));
  rp.launches += 2;
}
template <int H>
void launch_repulse_tc(RowPlan& rp, cudaStream_t s, int cur, bool dependent) {
  static_assert(H <= 8, "the tensor form takes ndim <= 16");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)rp.rep_ctas); cfg.blockDim = dim3(kT2Threads);
  cfg.dynamicSmemBytes = T2Smem::kTotal; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = dependent ? 1 : 0;
  TL_CUDA(cudaLaunchKernelEx(&cfg, repulse_tc2_kernel<H>, rp.dv, t2_image(rp), cur, rp.tc_cpi));
}

template <int H, int kRing> constexpr size_t kWalkSmem = (size_t)(kBlockRows / 32) * Ring<H, kRing>::kWarpBytes;

// The overlap of launch_pass: two CTAs of the two-GEMM pass and one walk CTA (either ring) share an SM's 233,472 bytes
// of shared memory.  The system reserves 1 KiB per CTA; kWalkStaticSmem is the walk's static shared memory with that
// reserve, as cuobjdump -res-usage reports it (tests/test_resource_budget.py checks it and the register caps).
constexpr size_t kSmPerSm = 233472, kSmReserved = 1024, kWalkStaticSmem = 1152;
static_assert(2 * (T2Smem::kTotal + kSmReserved) + kWalkSmem<8, 4> + kWalkStaticSmem <= kSmPerSm &&
              2 * (T2Smem::kTotal + kSmReserved) + kWalkSmem<8, 8> + kWalkStaticSmem <= kSmPerSm,
              "two repulse_tc2_kernel CTAs and a spring_kernel CTA no longer fit in one SM's shared memory");

// the spring / MAE launches of one rank (deep ring when the rank owns few rows)
template <int H>
void launch_spring(const RowPlan& rp, cudaStream_t s, int cur, unsigned e_spring, int ctas);
template <int H>
void launch_mae(const RowPlan& rp, cudaStream_t s, int nxt, unsigned e_spring, unsigned e_mae);

// The pass of one rank over positions buffer `cur`: the tensor form's image, the repulsion pass (the FP32 difference form,
// the tensor form, or both when the device picks per iteration), the spring walk, and combine_kernel, which signals the
// next epoch.  overlap: the spring walk runs beside the repulsion pass; otherwise the kernels run one after another.
// ev: null, or events 0..3 of row_time_kernels.
template <int H>
void launch_pass(RowPlan& rp, cudaStream_t s, int cur, cudaEvent_t* ev, bool overlap) {
  RowDev& dv = rp.dv;
  const unsigned e_prev = rp.epoch;          // the epoch every rank reached when the iteration before (and its check) ended
  if (ev) TL_CUDA(cudaEventRecord(ev[0], s));
  if constexpr (H <= 8) {                    // the tensor form exists for ndim <= 16 only
    if (rp.tc_form) launch_image_tc<H>(rp, s, cur, e_prev);
  }
  if (overlap) {
    // The walk first: its CTAs announce themselves at once (griddepcontrol.launch_dependents), which lets the
    // repulsion grid - launched as a programmatic dependent, it has no data dependence on the walk - fill the
    // rest of the chip while the walk's warps are already resident.  Under the two-GEMM pass the walk is one CTA per
    // SM (walk_ctas), each walking several row blocks: two pass CTAs fit beside it (static_assert above), and its warps,
    // the older ones on the SM, keep their issue priority - launched after the pass, the walk's latency chain got a
    // fraction of the issue slots and ended 0.8 ms after the pass (cfg4).  (Launched from two streams the repulsion grid
    // usually won the race for the SMs and the walk ran after it.)
    launch_spring<H>(rp, s, cur, e_prev, rp.walk_ctas);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)rp.f32_ctas); cfg.blockDim = dim3((unsigned)rp.f32_threads);
    cfg.dynamicSmemBytes = rp.f32_smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (!rp.tc_form || dv.adaptive) {
      TL_CUDA(cudaLaunchKernelEx(&cfg, (RepulseFn)rp.rep_fn, dv, cur, e_prev));
      rp.launches += dv.adaptive ? 1 : 0;
    }
    if constexpr (H <= 8) { if (rp.tc_form) launch_repulse_tc<H>(rp, s, cur, true); }
  } else {
    if (!rp.tc_form || dv.adaptive) {
      ((RepulseFn)rp.rep_fn)<<<rp.f32_ctas, rp.f32_threads, rp.f32_smem, s>>>(dv, cur, e_prev);
      rp.launches += dv.adaptive ? 1 : 0;
    }
    if constexpr (H <= 8) { if (rp.tc_form) launch_repulse_tc<H>(rp, s, cur, false); }
    if (ev) TL_CUDA(cudaEventRecord(ev[1], s));
    launch_spring<H>(rp, s, cur, e_prev, dv.rows / kBlockRows);
    if (ev) TL_CUDA(cudaEventRecord(ev[2], s));
  }
  combine_kernel<H><<<dv.rows / kBlockRows, kBlockRows, 0, s>>>(dv, rp.prm, cur, ++rp.epoch);
  if (ev) TL_CUDA(cudaEventRecord(ev[3], s));
  rp.launches += 3;
}

// ctl_kernel raises FitState::snapshot when its check improved the best state, and snap_kernel copies the positions
// while it is raised.  The flag is cleared after every snap launch: once a fit has stopped, ctl_kernel returns at
// once and a raised flag would stay raised, so the snap launches of the iterations the host had already enqueued
// would copy the position buffer of their own parity over the best state - for every second of them the positions of
// the iteration before the last one.  How many such launches there are depends on host timing, so the best positions
// (and the hold-out sums scored on them) of a fit that stopped early depended on it.
void clear_snapshot(const RowPlan& rp, cudaStream_t s) {
  TL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(rp.state) + offsetof(FitState, snapshot), 0, sizeof(int), s));
}

// One iteration of one rank: the pass, then on check and finite-check iterations the edge MAE, the controller and the
// best-state snapshot.
template <int H>
void launch_iteration(RowPlan& rp, cudaStream_t s, cudaEvent_t* ev /* 7 events or null */, bool overlap) {
  RowDev& dv = rp.dv;
  const int t = rp.iter_launched;
  const int cur = t & 1, nxt = cur ^ 1;
  const bool check = is_check_iter(t, rp.prm), fin = ((t + 1) % 10 == 0);
  launch_pass<H>(rp, s, cur, ev, overlap);
  if (check || fin) {
    const unsigned e_iter = rp.epoch;
    const unsigned e_mae = ++rp.epoch;
    launch_mae<H>(rp, s, nxt, e_iter, e_mae);
    if (ev) TL_CUDA(cudaEventRecord(ev[4], s));
    ctl_kernel<<<1, 256, 0, s>>>(dv, rp.prm, check ? 1 : 0, fin ? 1 : 0, e_mae);
    if (ev) TL_CUDA(cudaEventRecord(ev[5], s));
    snap_kernel<<<148, 256, 0, s>>>(dv, nxt);
    if (ev) TL_CUDA(cudaEventRecord(ev[6], s));
    clear_snapshot(rp, s);
    rp.launches += 3;
  }
  TL_CUDA(cudaGetLastError());
  rp.iter_launched = t + 1;
}

template <int H>
void launch_spring(const RowPlan& rp, cudaStream_t s, int cur, unsigned e_spring, int ctas) {
  if (rp.deep_ring) spring_kernel<H, 8><<<ctas, kBlockRows, kWalkSmem<H, 8>, s>>>(rp.dv, rp.prm, cur, e_spring);
  else spring_kernel<H, 4><<<ctas, kBlockRows, kWalkSmem<H, 4>, s>>>(rp.dv, rp.prm, cur, e_spring);
}
template <int H>
void launch_mae(const RowPlan& rp, cudaStream_t s, int nxt, unsigned e_spring, unsigned e_mae) {
  const int ctas = rp.dv.rows / kBlockRows;
  if (rp.deep_ring) mae_kernel<H, 8><<<ctas, kBlockRows, kWalkSmem<H, 8>, s>>>(rp.dv, nxt, e_spring, e_mae);
  else mae_kernel<H, 4><<<ctas, kBlockRows, kWalkSmem<H, 4>, s>>>(rp.dv, nxt, e_spring, e_mae);
}

void launch_one(RowPlan& rp, cudaStream_t s, cudaEvent_t* ev = nullptr) {
  dispatch_h(row_h(rp.dv.D), [&](auto h) { launch_iteration<decltype(h)::value>(rp, s, ev, rp.overlap && !ev); });
}

// The form of the repulsion pass.  Policy: 11, the two-GEMM tensor-core pass (rowblock_tc2.cuh), for ndim 5..16 and
// adaptive (see below); 5, the FP32 difference form (repulse_kernel), below ndim 5 and above 16.  Measured on B200 (ms per
// repulsion pass, forms 11 / 5): ndim 16, 100k: 7.5 / 16.8; ndim 12, 40k: 1.24 / 2.32; ndim 10, 10k: 0.16 / 0.23; ndim 6,
// 30k: 0.69 / 0.75.  The two-GEMM form costs the same at every ndim (K is padded to 16 coordinates); the difference form's
// cost falls with ndim and takes over below ndim 5.  TOPOLOW_REP_VARIANT=5 or 11 runs that form in every iteration.
template <int H>
void configure_repulse(RowPlan& rp, int sms) {
  const char* ev = std::getenv("TOPOLOW_REP_VARIANT");
  int form = (H >= 3 && H <= 8) ? 11 : 5;
  if (ev) {
    if (std::strcmp(ev, "5") == 0) form = 5;
    else if (std::strcmp(ev, "11") == 0) form = 11;
    else throw BadArg("TOPOLOW_REP_VARIANT takes 5 (FP32 difference form) or 11 (two-GEMM tensor-core form) in row-block mode");
    // ndim 17..32: the two-GEMM pass pads K to 16 coordinates; only the difference form is built, and asking for the
    // other form is an error, not a silent substitute
    if (H > 8 && form != 5) throw BadArg("ndim > 16 runs only the FP32 difference form (TOPOLOW_REP_VARIANT=5) in row-block mode");
  }
  rp.rep_form = form;
  rp.tc_form = form == 11;
  if constexpr (H <= 8) if (rp.tc_form) {
    rp.dv.rparts = 3 * rp.dv.chunks;
    TL_CUDA(cudaFuncSetAttribute(repulse_tc2_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2Smem::kTotal));
    TL_CUDA(cudaFuncSetAttribute(repulse_tc2_kernel<H>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // The occupancy API answers 1 for a kernel that allocates tensor memory (it cannot know how many of the 512 columns
    // tcgen05.alloc will ask for); registers, shared memory and the 256 columns a CTA takes all allow two, and the work
    // split does not depend on how many CTAs are resident at once.
    const int per_sm = 2;
    const long long pairs = (long long)(rp.dv.rows / kRowTile) * rp.dv.chunks;
    rp.tc_cpi = (int)std::max<long long>(1, std::min<long long>(rp.dv.chunks, pairs / (6ll * sms * per_sm)));
    const long long items = (long long)(rp.dv.rows / kRowTile) * ((rp.dv.chunks + rp.tc_cpi - 1) / rp.tc_cpi);
    rp.rep_ctas = (int)std::min<long long>((long long)sms * per_sm, std::max<long long>(items, 1));
    rp.rep_items = items;
  }
  // the FP32 difference form: two rows per thread, two partners per trip; ndim 17..32 one row per thread (two rows and
  // their accumulators alone are 4 H float2)
  RepulseFn fn;
  int threads;
  if constexpr (H <= 8) { fn = repulse_kernel<H, 2, 2, 128>; threads = kRowTile / 2; }
  else { fn = repulse_kernel<H, 1, kRepUnrollWide, kRepRegsWide>; threads = kRowTile; }
  const size_t smem = (size_t)kStages * kStageJ * Row<H>::kStride * sizeof(float);
  cudaFuncAttributes fa;
  TL_CUDA(cudaFuncGetAttributes(&fa, (const void*)fn));
  // the static shared memory counts against the same 48 KB default (ndim 32: 48 KB of stages + item_s)
  if (smem + fa.sharedSizeBytes > 48 * 1024) TL_CUDA(cudaFuncSetAttribute((const void*)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  TL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
  if (per_sm < 1) per_sm = 1;
  const long long items = (long long)(rp.dv.rows / kRowTile) * rp.dv.chunks;
  rp.f32_ctas = (int)std::min<long long>((long long)sms * per_sm, std::max<long long>(items, 1));
  rp.f32_smem = smem; rp.f32_threads = threads;
  rp.rep_fn = (void*)fn;
  if (!rp.tc_form) { rp.rep_ctas = rp.f32_ctas; rp.rep_items = items; }
  // The policy's tensor form is adaptive: the device picks the form of every iteration (image_tc_kernel's probe) and
  // the host launches both kernels.  A form asked for by name (TOPOLOW_REP_VARIANT) runs unconditionally.
  rp.dv.adaptive = (rp.tc_form && !ev) ? 1 : 0;
  if (const char* ea = std::getenv("TOPOLOW_ADAPTIVE")) rp.dv.adaptive = (rp.tc_form && std::atoi(ea) != 0) ? 1 : 0;
  rp.dv.series = rp.dv.adaptive;     // not adaptive: the series form only on request (it is exact only for pairs farther than 0.1 apart)
  if (const char* es = std::getenv("TOPOLOW_TC_SERIES")) rp.dv.series = std::atoi(es) != 0 ? 1 : 0;
  rp.dv.probe_k = (int)std::min<long long>(64, std::max<long long>(4, (262144 + rp.dv.n - 1) / std::max(rp.dv.n, 1)));
  // Break-even, measured at cfg4 (ndim 16): the fix-ups cost about 4.7 s x (near fraction) per pass over 1e10 one-sided pairs,
  // the difference form 9 ms more than the tensor form: near fraction 2e-3; half of that is the limit, scaled with ndim
  // (the difference form's cost falls with ndim, the tensor form's does not).
  const double p_lim = 1.25e-4 * H;
  if (const char* el = std::getenv("TOPOLOW_NEAR_LIMIT")) { rp.near_limit = std::atof(el); } else rp.near_limit = p_lim;
  rp.dv.probe_limit = (unsigned)((double)rp.dv.probe_k * (double)rp.dv.n * rp.near_limit);
  rp.sm_count = sms;
  rp.overlap = true;   // measured on B200 at cfg4: one rank of 8 2.61 -> 2.38 ms, of 2 9.11 -> 8.99, one GPU 18.29 -> 18.11; cfg3 0.47 -> 0.29
  if (const char* eo = std::getenv("TOPOLOW_OVERLAP")) rp.overlap = std::atoi(eo) != 0;
  // spring / MAE walk: the deep ring needs more than the default 48 KB of dynamic shared memory
  rp.deep_ring = rp.dv.rows / kBlockRows <= 2 * sms;
  rp.walk_ctas = rp.tc_form ? std::min(rp.dv.rows / kBlockRows, sms) : rp.dv.rows / kBlockRows;
  TL_CUDA(cudaFuncSetAttribute(spring_kernel<H, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWalkSmem<H, 8>));
  TL_CUDA(cudaFuncSetAttribute(mae_kernel<H, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWalkSmem<H, 8>));
  if constexpr (kWalkSmem<H, 4> > 48 * 1024) {   // 128-byte ring rows (ndim 17..32): the 4-deep ring needs it too
    TL_CUDA(cudaFuncSetAttribute(spring_kernel<H, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWalkSmem<H, 4>));
    TL_CUDA(cudaFuncSetAttribute(mae_kernel<H, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWalkSmem<H, 4>));
  }
}

}  // namespace

RowPlan* row_create(const topolow_problem& pb, const topolow_params& pr, int rank, int n_ranks) {
  validate(pb, pr);
  if (n_ranks < 1 || n_ranks > kMaxShards || rank < 0 || rank >= n_ranks) throw BadArg("rank / n_ranks out of range");
  if (pb.ndim > 32) throw BadArg("row-block mode supports ndim <= 32 (the replay mode takes any ndim)");
  if (pb.n >= (1ll << 30)) throw BadArg("n out of range");
  TL_CUDA(cudaSetDevice(pr.device));
  keep_pool_memory(pr.device);
  int sm_count = 0;
  TL_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, pr.device));   // (cudaGetDeviceProperties costs milliseconds)
  std::unique_ptr<RowPlan> rp(new RowPlan());
  rp->device = pr.device;
  rp->n = pb.n; rp->E = pb.n_edges;
  rp->prm = FitParams{pr.n_iter, pr.k0, pr.cooling_rate, pr.c_repulsion, pr.relative_epsilon, pr.convergence_window,
                      pr.convergence_check_freq};
  RowDev& dv = rp->dv;
  dv.n = (int)pb.n; dv.D = pb.ndim; dv.Dp = (pb.ndim + 3) / 4 * 4;
  dv.G = n_ranks; dv.rank = rank;
  const int tiles = (int)((pb.n + kRowTile - 1) / kRowTile);
  dv.slots = tiles * kRowTile;
  const int t0 = (int)((long long)tiles * rank / n_ranks), t1 = (int)((long long)tiles * (rank + 1) / n_ranks);
  dv.row0 = t0 * kRowTile; dv.rows = (t1 - t0) * kRowTile;
  if (tiles < n_ranks) throw BadArg("too few points for this many ranks (every rank needs at least 256 rows)");
  dv.chunks = (int)((pb.n + kChunk - 1) / kChunk);
  dv.rparts = dv.chunks;
  dv.cap_rows = align_up((size_t)dv.slots, kChunk);
  dv.pairs_per_iter = (unsigned long long)pb.n * (unsigned long long)(pb.n - 1) / 2ull;
  dv.seed = pr.seed;
  dv.no_wait = std::getenv("TOPOLOW_IGNORE_PEERS") ? 1 : 0;
  TL_CUDA(cudaStreamCreate(&rp->stream));
  TL_CUDA(cudaEventCreate(&rp->ev0));
  TL_CUDA(cudaEventCreate(&rp->ev1));
  PhaseTimer pt(rp->stream);
  // relabelling: a fixed pseudo-random permutation (decorrelates the caller's row order from the row
  // blocks and from the order a row visits its partners in)
  rp->slot_of_point = random_permutation(pb.n, kRowLayoutSeed);
  pt.mark("rows: relabelling");

  // ---- shared block ----
  const size_t pos_bytes = 2 * dv.cap_rows * dv.Dp * sizeof(float);
  rp->off_red = align_up(pos_bytes, 256);
  rp->off_flags = align_up(rp->off_red + (size_t)(dv.slots / kBlockRows) * 4 * sizeof(double), 256);
  rp->shared_bytes = align_up(rp->off_flags + (size_t)kMaxShards * kFlagStride * sizeof(unsigned), 256);
  TL_CUDA(cudaMalloc((void**)&rp->shared, rp->shared_bytes));
  TL_CUDA(cudaMemset(rp->shared, 0, rp->shared_bytes));
  set_self_pointers(*rp);
  pt.mark("rows: shared block");

  // ---- points ----
  {
    std::vector<float> hp(dv.cap_rows * dv.Dp, 0.f), hd(dv.slots, 0.f);
    for (int64_t i = 0; i < pb.n; ++i) {
      const size_t sl = rp->slot_of_point[i];
      for (int d = 0; d < pb.ndim; ++d) hp[sl * dv.Dp + d] = (float)pb.initial_positions[(size_t)d * pb.n + i];
      hd[sl] = (float)((double)pb.degrees[i] + 1.0);
    }
    pool_alloc(rp->best, hp.size() * sizeof(float));
    pool_alloc(rp->dp1, hd.size() * sizeof(float));
    pool_alloc(rp->rpart, (size_t)(pb.ndim <= 16 ? 3 : 1) * dv.chunks * std::max(dv.rows, 1) * dv.Dp * sizeof(float));   // 3: the two-GEMM form
    pool_alloc(rp->tc_buf, dv.cap_rows * (size_t)(16 + 16 + 4 + 4 + 16 + 32 + 16) * sizeof(float));
    pool_alloc(rp->xs, (size_t)std::max(dv.rows, 1) * dv.Dp * sizeof(float));
    pool_alloc(rp->state, sizeof(FitState));
    pool_alloc(rp->trace, sizeof(double) * std::max(pr.n_iter, 1));
    pool_alloc(rp->counters, 8 * sizeof(unsigned));
    pool_ready();
    TL_CUDA(cudaMemcpy(rp->shared, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice));
    TL_CUDA(cudaMemcpy(rp->best, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice));
    TL_CUDA(cudaMemcpy(rp->dp1, hd.data(), hd.size() * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<double> tr(std::max(pr.n_iter, 1), NAN);
    TL_CUDA(cudaMemcpy(rp->trace, tr.data(), tr.size() * sizeof(double), cudaMemcpyHostToDevice));
    TL_CUDA(cudaMemset(rp->counters, 0, 8 * sizeof(unsigned)));
    // centre of the tensor form's image: the centroid of the initial positions, summed in point order (the same on
    // every rank, fixed for the fit; the map stays about where it starts, and a map that wanders only makes more
    // pairs take the difference form)
    for (int d = 0; d < 16; ++d) dv.centre[d] = 0.f;
    for (int d = 0; d < std::min(pb.ndim, 16); ++d) {   // ndim > 16 runs the difference form, which has no centre
      double sum = 0.0;
      for (int64_t i = 0; i < pb.n; ++i) sum += pb.initial_positions[(size_t)d * pb.n + i];
      const double c = sum / (double)pb.n;
      dv.centre[d] = std::isfinite(c) ? (float)c : 0.f;
    }
    FitState st;
    state_init(st, rp->prm);
    TL_CUDA(cudaMemcpy(rp->state, &st, sizeof st, cudaMemcpyHostToDevice));
  }
  pt.mark("rows: points");
  dv.best = rp->best; dv.dp1 = rp->dp1; dv.rpart = rp->rpart; dv.xs = rp->xs;
  dv.state = rp->state; dv.trace = rp->trace;
  dv.counters = rp->counters;
  TL_CUDA(cudaHostAlloc((void**)&rp->h_flag, 2 * sizeof(int), cudaHostAllocMapped));
  rp->h_flag[0] = 0; rp->h_flag[1] = 0;
  TL_CUDA(cudaHostGetDevicePointer((void**)&rp->d_flag, (void*)rp->h_flag, 0));
  dv.host_flag = rp->d_flag;

  if (dv.rows > 0) build_records(*rp, pb);
  if (pb.n_holdout > 0) {
    if (!pb.holdout_i || !pb.holdout_j || !pb.holdout_truth) throw BadArg("hold-out arrays are required when n_holdout > 0");
    rp->n_holdout = pb.n_holdout;
    rp->hold_i.assign(pb.holdout_i, pb.holdout_i + pb.n_holdout);
    rp->hold_j.assign(pb.holdout_j, pb.holdout_j + pb.n_holdout);
    rp->hold_truth.assign(pb.holdout_truth, pb.holdout_truth + pb.n_holdout);
  }
  pt.mark("rows: records + hold-out");
  if (dv.rows > 0) dispatch_h(row_h(dv.D), [&](auto h) { configure_repulse<decltype(h)::value>(*rp, sm_count); });
  pt.mark("rows: kernel attributes");
  TL_CUDA(cudaDeviceSynchronize());
  pt.mark("rows: device synchronize");
  rp->attached = (n_ranks == 1);
  return rp.release();
}

void row_destroy(RowPlan* rp) { delete rp; }

size_t row_handle_bytes() { return sizeof(RowHandle); }

void row_export(RowPlan& rp, void* blob) {
  DeviceScope on(rp.device);
  RowHandle h{};
  TL_CUDA(cudaIpcGetMemHandle(&h.mem, rp.shared));
  h.rank = rp.dv.rank; h.n_ranks = rp.dv.G; h.slots = rp.dv.slots; h.Dp = rp.dv.Dp; h.layout = rp.shared_bytes;
  std::memcpy(blob, &h, sizeof h);
}

void row_attach(RowPlan& rp, const void* blobs, int n_blobs) {
  DeviceScope on(rp.device);
  if (n_blobs != rp.dv.G) throw BadArg("one handle per rank is required");
  const RowHandle* hs = static_cast<const RowHandle*>(blobs);
  for (int q = 0; q < n_blobs; ++q) {
    RowHandle h;
    std::memcpy(&h, hs + q, sizeof h);
    if (h.rank != q || h.n_ranks != rp.dv.G || h.slots != rp.dv.slots || h.Dp != rp.dv.Dp || h.layout != rp.shared_bytes)
      throw BadArg("the ranks of a sharded map must be created from the same problem");
    if (q == rp.dv.rank) continue;
    void* base = nullptr;
    TL_CUDA(cudaIpcOpenMemHandle(&base, h.mem, cudaIpcMemLazyEnablePeerAccess));
    rp.peer_base[q] = base; rp.peer_ipc[q] = true;
    set_peer_pointers(rp, q, static_cast<char*>(base));
  }
  rp.attached = true;
}

void row_attach_local(RowPlan* const* plans, int n) {
  if (n < 1 || n > kMaxShards) throw BadArg("number of replicas out of range");
  for (int a = 0; a < n; ++a) {
    RowPlan& pa = *plans[a];
    if (pa.dv.G != n || pa.dv.rank != a) throw BadArg("replicas must be passed in rank order");
    if (pa.dv.slots != plans[0]->dv.slots || pa.dv.Dp != plans[0]->dv.Dp) throw BadArg("the ranks of a sharded map must be created from the same problem");
    DeviceScope on(pa.device);
    for (int b = 0; b < n; ++b) {
      if (a == b) continue;
      RowPlan& pb = *plans[b];
      if (pb.device != pa.device) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(pb.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) TL_CUDA(e);
        cudaGetLastError();
      }
      pa.peer_base[b] = pb.shared; pa.peer_ipc[b] = false;
      set_peer_pointers(pa, b, pb.shared);
    }
    pa.attached = true;
  }
}

static void check_runnable(const RowPlan& rp) {
  if (!rp.attached) throw BadArg("the replicas of a sharded map must be attached before it runs");
}

double row_run(RowPlan& rp, int n_iters, cudaStream_t stream_in, topolow_interrupt_fn poll, void* user, bool* interrupted) {
  check_runnable(rp);
  TL_CUDA(cudaSetDevice(rp.device));
  cudaStream_t s = stream_in ? stream_in : rp.stream;
  TL_CUDA(cudaEventRecord(rp.ev0, s));
  int left = std::min(n_iters, std::max(0, rp.prm.n_iter - rp.iter_launched));
  int since_sync = 0;
  while (left > 0) {
    if (rp.h_flag[0]) break;
    if (poll && since_sync == 0 && poll(user)) { if (interrupted) *interrupted = true; break; }
    launch_one(rp, s);
    --left;
    if (++since_sync >= 50) {             // the reference's interrupt interval (src/optimization.cpp:364)
      since_sync = 0;
      if (poll) TL_CUDA(cudaStreamSynchronize(s));
    }
  }
  TL_CUDA(cudaEventRecord(rp.ev1, s));
  TL_CUDA(cudaEventSynchronize(rp.ev1));
  float ms = 0.f;
  TL_CUDA(cudaEventElapsedTime(&ms, rp.ev0, rp.ev1));
  rp.total_ms += ms;
  return ms;
}

bool row_run_windows(RowPlan& rp, const std::function<bool()>& stop) {
  check_runnable(rp);
  TL_CUDA(cudaSetDevice(rp.device));
  constexpr int kWindow = 5;                  // iterations per window; two windows in flight
  cudaStream_t s = rp.stream;
  EventGuard win[2];
  // (returns true when `stop` fired before `e` completed)
  auto wait = [&](cudaEvent_t e) {
    while (true) {
      const cudaError_t q = cudaEventQuery(e);
      if (q == cudaSuccess) return false;
      if (q != cudaErrorNotReady) TL_CUDA(q);
      if (stop()) return true;
      std::this_thread::sleep_for(std::chrono::microseconds(200));
    }
  };
  TL_CUDA(cudaEventRecord(rp.ev0, s));
  int left = std::max(0, rp.prm.n_iter - rp.iter_launched);
  bool cut = false;
  for (int w = 0; left > 0 && !rp.h_flag[0]; ++w) {
    if (w >= 2 ? wait(win[w & 1]) : (w == 1 && stop())) { cut = true; break; }   // window w - 2 has ended
    const int c = std::min(left, kWindow);
    for (int i = 0; i < c; ++i) launch_one(rp, s);
    left -= c;
    TL_CUDA(cudaEventRecord(win[w & 1], s));
  }
  TL_CUDA(cudaEventRecord(rp.ev1, s));
  if (!cut) wait(rp.ev1);                     // a stop request now lets the queued iterations finish the fit
  if (cudaPeekAtLastError() == cudaErrorNotReady) cudaGetLastError();
  TL_CUDA(cudaEventSynchronize(rp.ev1));
  float ms = 0.f;
  TL_CUDA(cudaEventElapsedTime(&ms, rp.ev0, rp.ev1));
  rp.total_ms += ms;
  return cut && !rp.h_flag[0];                // a fit that converged or failed on its own was not cut short
}

double row_run_local(RowPlan* const* plans, int n, int n_iters) {
  for (int a = 0; a < n; ++a) check_runnable(*plans[a]);
  bool same_device = true;
  for (int a = 1; a < n; ++a) same_device = same_device && plans[a]->device == plans[0]->device;
  RowPlan& p0 = *plans[0];
  int left = std::min(n_iters, std::max(0, p0.prm.n_iter - p0.iter_launched));
  TL_CUDA(cudaSetDevice(p0.device));
  TL_CUDA(cudaEventRecord(p0.ev0, p0.stream));
  if (same_device) {
    // lock step on ONE stream: rank after rank, phase after phase, so that every wait finds its epoch reached
    cudaStream_t s = p0.stream;
    for (int a = 0; a < n; ++a) TL_CUDA(cudaStreamSynchronize(plans[a]->stream));
    while (left > 0) {
      if (p0.h_flag[0]) break;
      const int t = p0.iter_launched;
      const int cur = t & 1, nxt = cur ^ 1;
      const bool check = is_check_iter(t, p0.prm), fin = ((t + 1) % 10 == 0);
      for (int a = 0; a < n; ++a) {
        RowPlan& rp = *plans[a];
        dispatch_h(row_h(rp.dv.D), [&](auto h) { launch_pass<decltype(h)::value>(rp, s, cur, nullptr, false); });
        rp.iter_launched = t + 1;
      }
      if (check || fin) {
        for (int a = 0; a < n; ++a) {
          RowPlan& rp = *plans[a];
          dispatch_h(row_h(rp.dv.D), [&](auto h) {
            constexpr int H = decltype(h)::value;
            const unsigned e_iter = rp.epoch;
            launch_mae<H>(rp, s, nxt, e_iter, ++rp.epoch);
          });
          rp.launches += 1;
        }
        for (int a = 0; a < n; ++a) {
          RowPlan& rp = *plans[a];
          ctl_kernel<<<1, 256, 0, s>>>(rp.dv, rp.prm, check ? 1 : 0, fin ? 1 : 0, rp.epoch);
          snap_kernel<<<148, 256, 0, s>>>(rp.dv, nxt);
          clear_snapshot(rp, s);
          rp.launches += 2;
        }
      }
      TL_CUDA(cudaGetLastError());
      --left;
      if ((t + 1) % 50 == 0) TL_CUDA(cudaStreamSynchronize(s));
    }
    TL_CUDA(cudaEventRecord(p0.ev1, s));
  } else {
    while (left > 0) {
      if (p0.h_flag[0]) break;
      for (int a = 0; a < n; ++a) {
        TL_CUDA(cudaSetDevice(plans[a]->device));
        launch_one(*plans[a], plans[a]->stream);
      }
      --left;
    }
    for (int a = 1; a < n; ++a) { TL_CUDA(cudaSetDevice(plans[a]->device)); TL_CUDA(cudaStreamSynchronize(plans[a]->stream)); }
    TL_CUDA(cudaSetDevice(p0.device));
    TL_CUDA(cudaEventRecord(p0.ev1, p0.stream));
  }
  TL_CUDA(cudaEventSynchronize(p0.ev1));
  float ms = 0.f;
  TL_CUDA(cudaEventElapsedTime(&ms, p0.ev0, p0.ev1));
  for (int a = 0; a < n; ++a) plans[a]->total_ms += ms;
  return ms;
}

void row_time_kernels(RowPlan& rp, int n_iters, double* out, int cap) {
  check_runnable(rp);
  TL_CUDA(cudaSetDevice(rp.device));
  double acc[7] = {0, 0, 0, 0, 0, 0, 0};
  int done = 0;
  std::vector<EventGuard> evs(7);
  cudaEvent_t ev[7];
  for (int i = 0; i < 7; ++i) ev[i] = evs[i];
  int left = std::min(n_iters, std::max(0, rp.prm.n_iter - rp.iter_launched));
  while (left-- > 0 && !rp.h_flag[0]) {
    const int t = rp.iter_launched;
    const bool extra = is_check_iter(t, rp.prm) || ((t + 1) % 10 == 0);
    launch_one(rp, rp.stream, ev);     // in order on one stream: every kernel is timed alone
    TL_CUDA(cudaStreamSynchronize(rp.stream));
    float ms = 0.f;
    TL_CUDA(cudaEventElapsedTime(&ms, ev[0], ev[1])); acc[0] += ms;
    TL_CUDA(cudaEventElapsedTime(&ms, ev[1], ev[2])); acc[1] += ms;
    TL_CUDA(cudaEventElapsedTime(&ms, ev[2], ev[3])); acc[6] += ms;
    if (extra) {
      TL_CUDA(cudaEventElapsedTime(&ms, ev[3], ev[4])); acc[2] += ms;
      TL_CUDA(cudaEventElapsedTime(&ms, ev[4], ev[5])); acc[3] += ms;
      TL_CUDA(cudaEventElapsedTime(&ms, ev[5], ev[6])); acc[4] += ms;
      acc[5] += 1.0;
    }
    ++done;
  }
  const double v[7] = {done ? acc[0] / done : 0.0, done ? acc[1] / done : 0.0, acc[5] > 0 ? acc[2] / acc[5] : 0.0,
                       acc[5] > 0 ? acc[3] / acc[5] : 0.0, acc[5] > 0 ? acc[4] / acc[5] : 0.0, acc[5],
                       done ? acc[6] / done : 0.0};
  for (int i = 0; i < cap && i < 7; ++i) out[i] = v[i];
}

void row_result(RowPlan& rp, topolow_result& res, bool interrupted) {
  TL_CUDA(cudaSetDevice(rp.device));
  TL_CUDA(cudaStreamSynchronize(rp.stream));
  FitState st;
  TL_CUDA(cudaMemcpy(&st, rp.state, sizeof st, cudaMemcpyDeviceToHost));
  const RowDev& dv = rp.dv;
  if (res.positions) {
    std::vector<float> hp((size_t)dv.slots * dv.Dp);
    TL_CUDA(cudaMemcpy(hp.data(), rp.best, hp.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < rp.n; ++i) {
      const size_t sl = rp.slot_of_point[i];
      for (int d = 0; d < dv.D; ++d) res.positions[(size_t)d * rp.n + i] = (double)hp[sl * dv.Dp + d];
    }
  }
  res.converged = st.converged;
  res.iterations = st.best_iter;     // src/optimization.cpp:368-381: always the best snapshot
  res.final_mae = st.best_mae;
  res.final_k = st.best_k;
  res.iterations_run = st.iter;
  res.pair_updates = (int64_t)st.pair_updates;
  res.device_ms = rp.total_ms;
  if (dv.adaptive) {
    unsigned c[8];
    TL_CUDA(cudaMemcpy(c, rp.counters, sizeof c, cudaMemcpyDeviceToHost));
    rp.tensor_iters = (int64_t)c[7];
    if (std::getenv("TOPOLOW_DEBUG"))
      std::fprintf(stderr, "[topolow] rows: %lld of %d iterations ran the tensor form (probe: %d partners per row, limit %u near pairs)\n",
                   (long long)rp.tensor_iters, st.iter, dv.probe_k, dv.probe_limit);
  }
  res.fail_iter = st.fail_iter;
  res.status = TOPOLOW_OK;
  res.message[0] = 0;
  res.holdout_sum_abs = 0.0; res.holdout_count = 0;
  if (st.status == 2) {
    res.status = TOPOLOW_ERR_NONFINITE;
    std::snprintf(res.message, sizeof res.message, "Numerical instability at iteration %d. Reduce k0 or c_repulsion.", st.fail_iter);
  } else if (st.status == 3) {
    res.status = TOPOLOW_ERR_CUDA;
    std::snprintf(res.message, sizeof res.message, "a peer replica of the sharded map did not arrive within 20 s");
  } else if (interrupted) {
    res.status = TOPOLOW_ERR_INTERRUPTED;
    std::snprintf(res.message, sizeof res.message, "interrupted");
  }
  if (res.status == TOPOLOW_OK && rp.n_holdout > 0 && res.positions &&
      topolow_holdout_errors(res.positions, rp.n, dv.D, rp.n_holdout, rp.hold_i.data(), rp.hold_j.data(), rp.hold_truth.data(),
                             &res.holdout_sum_abs, &res.holdout_count, rp.device) != TOPOLOW_OK)
    throw BadArg("hold-out cells out of range");
  if (res.trace_mae && rp.prm.n_iter > 0)
    TL_CUDA(cudaMemcpy(res.trace_mae, rp.trace, sizeof(double) * rp.prm.n_iter, cudaMemcpyDeviceToHost));
}

void row_info(const RowPlan& rp, int64_t* out, int cap) {
  const RowDev& dv = rp.dv;
  const int64_t v[18] = {dv.slots, dv.D, dv.Dp, dv.G, dv.rank, dv.row0, dv.rows, dv.chunks, rp.n_recs, rp.n_mrecs, rp.launches,
                         rp.h_flag ? rp.h_flag[1] : 0, rp.h_flag ? rp.h_flag[0] : 0,
                         (int64_t)(dv.G - 1) * dv.rows * dv.Dp * 4,   // position bytes this rank stores into its peers per iteration
                         rp.rep_items, rp.rep_ctas, rp.rep_form, rp.tensor_iters};
  for (int i = 0; i < cap && i < 18; ++i) out[i] = v[i];
}

}  // namespace tl

// ---------------------------------------------------------------------------------------------------
// C ABI (include/topolow_b200.h, topolow_shard_*)
// ---------------------------------------------------------------------------------------------------
struct topolow_shard { tl::RowPlan* rp; };

using namespace tl;

namespace {
template <class F>
int guarded(char* message, int32_t message_len, F&& f) {
  try {
    f();
    return TOPOLOW_OK;
  } catch (const BadArg& e) {
    set_msg(message, message_len, e.what());
    return TOPOLOW_ERR_BAD_ARG;
  } catch (const std::invalid_argument& e) {
    set_msg(message, message_len, e.what());
    return TOPOLOW_ERR_BAD_ARG;
  } catch (const CudaError& e) {
    set_msg(message, message_len, e.what());
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  } catch (const std::exception& e) {
    set_msg(message, message_len, e.what());
    return TOPOLOW_ERR_BAD_ARG;
  }
}
}  // namespace

extern "C" {

int topolow_shard_create(const topolow_problem* problem, const topolow_params* params, int32_t rank, int32_t n_ranks,
                         topolow_shard** shard_out, char* message, int32_t message_len) {
  if (!problem || !params || !shard_out) return TOPOLOW_ERR_BAD_ARG;
  *shard_out = nullptr;
  if (problem->n < 2) { set_msg(message, message_len, "Need at least 2 points for embedding"); return TOPOLOW_ERR_TOO_FEW_POINTS; }
  return guarded(message, message_len, [&] {
    RowPlan* rp = row_create(*problem, *params, rank, n_ranks);
    *shard_out = new topolow_shard{rp};
  });
}
int64_t topolow_shard_handle_bytes(void) { return (int64_t)row_handle_bytes(); }
int topolow_shard_export(topolow_shard* shard, void* handle_out) {
  if (!shard || !handle_out) return TOPOLOW_ERR_BAD_ARG;
  return guarded(nullptr, 0, [&] { row_export(*shard->rp, handle_out); });
}
int topolow_shard_attach(topolow_shard* shard, const void* handles, int32_t n_handles, char* message, int32_t message_len) {
  if (!shard || !handles) return TOPOLOW_ERR_BAD_ARG;
  return guarded(message, message_len, [&] { row_attach(*shard->rp, handles, n_handles); });
}
int topolow_shard_attach_local(topolow_shard* const* shards, int32_t n, char* message, int32_t message_len) {
  if (!shards || n < 1 || n > kMaxShards) return TOPOLOW_ERR_BAD_ARG;
  return guarded(message, message_len, [&] {
    RowPlan* plans[kMaxShards];
    for (int a = 0; a < n; ++a) { if (!shards[a]) throw BadArg("null shard"); plans[a] = shards[a]->rp; }
    row_attach_local(plans, n);
  });
}
int topolow_shard_run(topolow_shard* shard, int32_t n_iters, void* stream, double* ms_out) {
  if (!shard) return TOPOLOW_ERR_BAD_ARG;
  return guarded(nullptr, 0, [&] {
    const double ms = row_run(*shard->rp, n_iters, (cudaStream_t)stream, nullptr, nullptr, nullptr);
    if (ms_out) *ms_out = ms;
  });
}
int topolow_shard_run_local(topolow_shard* const* shards, int32_t n, int32_t n_iters, double* ms_out) {
  if (!shards || n < 1 || n > kMaxShards) return TOPOLOW_ERR_BAD_ARG;
  return guarded(nullptr, 0, [&] {
    RowPlan* plans[kMaxShards];
    for (int a = 0; a < n; ++a) { if (!shards[a]) throw BadArg("null shard"); plans[a] = shards[a]->rp; }
    const double ms = row_run_local(plans, n, n_iters);
    if (ms_out) *ms_out = ms;
  });
}
int topolow_shard_time_kernels(topolow_shard* shard, int32_t n_iters, double* out, int32_t cap) {
  if (!shard || !out) return TOPOLOW_ERR_BAD_ARG;
  return guarded(nullptr, 0, [&] { row_time_kernels(*shard->rp, n_iters, out, cap); });
}
int topolow_shard_result(topolow_shard* shard, topolow_result* result) {
  if (!shard || !result) return TOPOLOW_ERR_BAD_ARG;
  const int rc = guarded(result->message, sizeof result->message, [&] { row_result(*shard->rp, *result, false); });
  if (rc != TOPOLOW_OK) { result->status = rc; return rc; }
  return result->status;
}
int topolow_shard_info(const topolow_shard* shard, int64_t* out, int32_t cap) {
  if (!shard || !out) return TOPOLOW_ERR_BAD_ARG;
  row_info(*shard->rp, out, cap);
  return TOPOLOW_OK;
}
// slot_of_point of the row-block layout (a pure function of n): lets a checker restate the order rows
// are grouped and partners are visited in.
int topolow_shard_slot_order(int64_t n, int32_t* slot_of_point_out) {
  if (n < 1 || !slot_of_point_out) return TOPOLOW_ERR_BAD_ARG;
  const std::vector<int32_t> p = random_permutation(n, kRowLayoutSeed);
  std::memcpy(slot_of_point_out, p.data(), (size_t)n * sizeof(int32_t));
  return TOPOLOW_OK;
}
void topolow_shard_destroy(topolow_shard* shard) {
  if (!shard) return;
  row_destroy(shard->rp);
  delete shard;
}

}  // extern "C"
