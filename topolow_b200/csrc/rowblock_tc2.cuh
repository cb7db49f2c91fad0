// topolow_b200/csrc/rowblock_tc2.cuh - included by rowblock.cu after rowblock_tc.cuh, inside namespace tl::{anonymous}.
//
// Repulsion pass with BOTH contractions on the tensor cores - the structure of a fused attention kernel:
//   GEMM 1   S = d^2 / 2 for 128 rows x 32 partners                    (as in rowblock_tc.cuh: 3-pass TF32, norms in K)
//   FP32     w = (d + 0.01)^-3 per pair, read from and written back to the same TMEM columns (weights of near pairs 0)
//   GEMM 2   D2[128 x 32] += w[128 x 32] Y[32 partners x 32]            A operand from TMEM, Y = (x_0..x_15, 1, 0...): columns
//                                                                       0..15 collect sum_j w x_j, column 16 collects sum_j w
// and per chunk of 2048 partners the rows' sums come out as D2[0..15] - x_i D2[16].  The FP32 pipes are left with 7.6
// instructions per pair - one of them on the special-function unit when the weights can be computed by the series form
// (all pairs of the batch farther apart than 0.1; image_tc_kernel's probe decides per iteration, rowblock_tc.cuh), two
// (square root, reciprocal) otherwise.  Measured at cfg4 (ncu): 5.7 ms per pass, 75 % of the issue slots, FMA pipe 40 %,
// special-function unit 45 %, tensor-core unit 40 %.
//
// Precision of GEMM 2: w is used as TF32 (truncated by the tensor core) consistently in the sums of w x_j and of w, so
// the difference D2[0..15] - x_i D2[16] still telescopes.  The partner coordinates enter rounded to TF32 (2^-11 relative:
// a partner seen 0.01 away from where it is, at distances of 10, with independent signs over 100 000 partners) - the
// second pass over the remainders (kT2LoPass) costs a quarter more tensor instructions and changes nothing measurable.
// A weight carries a relative error of 2^-11 with random sign: noise far below the Jacobi / Gauss-Seidel difference.
//
// Issue rate: a stage is 22 tensor instructions and 9 bulk copies for 8192 pairs, and the FP32 side needs only ~0.4 us
// for them.  One lane doing all of it (with the loop wrappers the compiler puts around a warp-uniform instruction in
// divergent code) took 2 us per stage; hence two whole, converged warps - one issues the MMAs, one the copies - with
// elect.sync around the single-lane instructions.
//
// TMEM (256 columns per CTA, two CTAs per SM): S / w  [2 buffers][2 tiles][32] = 128, D2 [2 tiles][32] = 64 (one buffer: the
// consumers read a chunk's sums before the first GEMM 2 of the next chunk, once per 64 stages), and the rows' TF32 image
// -A_hi [2 tiles][24] = 48 and -A_lo of tile 0 in the last 16: eleven of the fourteen MMAs of a GEMM 1 take their A operand from tensor memory instead of reading
// 4 KB of shared memory each (the tensor pipe's operand fetch was its busiest part: 57 % of the cycles, and the consumers
// waited a fifth of their time for distances).

constexpr int kT2SJ = 32;            // partners per stage
constexpr int kT2Stages = 4;
constexpr int kT2Threads = 320;       // 8 consumer warps + the MMA warp + the copy warp
constexpr float kT2SeriesS = 0.005f;   // series form of the weight: pairs closer than 0.1 (d^2 / 2 < 0.005) are near pairs
constexpr bool kT2LoPass = false;     // second pass of GEMM 2 over the TF32 remainders of the partner coordinates (see below)

// The only A operand GEMM 1 reads from shared memory is the remainders of tile 1 (tile 0's and both tiles' -A_hi and norm
// columns are in tensor memory): 4 planes x 128 rows x 16 B.  At 61.6 KB per CTA two CTAs leave room on the SM for a
// CTA of the spring walk (rowblock.cu, launch_iteration).
struct T2Smem {
  static constexpr int kALo1 = 0;                                  // 4 planes x 128 rows x 16 B
  static constexpr int kATx = 4 * 128 * 16;                        // bytes landing per item
  static constexpr int kStage0 = kALo1 + kATx;
  static constexpr int kBHi = 0;                                   // 6 planes x 32 x 16 B   (GEMM 1, K-major over coordinates)
  static constexpr int kBLo = 6 * kT2SJ * 16;                      // 4 planes
  static constexpr int kYHi = kBLo + 4 * kT2SJ * 16;               // 8 partner-quads x 32 rows x 16 B (GEMM 2, K-major over partners)
  static constexpr int kYLo = kYHi + 8 * 32 * 16;                  // 8 partner-quads x 16 rows x 16 B
  static constexpr int kRows32 = kYLo + 8 * 16 * 16;               // 32 x 64 B (near pairs only)
  static constexpr int kStageBytes = kRows32 + kT2SJ * 64;
  static constexpr int kBars = kStage0 + kT2Stages * kStageBytes;
  static constexpr int kNumBars = 1 + 2 * kT2Stages + 8 + 1;       // a_full | full, empty per stage | tfull x 2, wfull x 2, d2full, d2empty, a_tmem, - | a_free
  static constexpr int kTmemPtr = kBars + kNumBars * 8;
  static constexpr int kTotal = kTmemPtr + 16;
  static constexpr int kStageTx = 4 * kT2SJ * 16 + kT2SJ * 16 + 4 * kT2SJ * 16 + 8 * 32 * 16 + (kT2LoPass ? 8 * 16 * 16 : 0) + kT2SJ * 64;
};

struct T2Image {
  TcImage a;      // the arrays of the one-GEMM form
  float* yhi;     // [cap_rows / 4][32][4]   row n of a partner quad: n < 16 coordinate n (TF32-rounded), n = 16: 1, else 0
  float* ylo;     // [cap_rows / 4][16][4]   the remainders of the coordinates
};

TL_D void tc_st8(unsigned taddr, const unsigned (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
TL_D void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
TL_D void tc_mma_tf32_ts(unsigned d_tmem, unsigned a_tmem, unsigned long long b_desc, unsigned idesc, unsigned accumulate) {
  asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p; }"
               ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
TL_D bool elect_one() {
  unsigned pred = 0;
  asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p; }" : "=r"(pred));
  return pred != 0;
}
TL_D float rsqrt_approx_ftz(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
TL_D float rcp_approx_ftz(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

constexpr unsigned kT2Idesc1 = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 13) | ((unsigned)(kT2SJ >> 3) << 17) | ((128u >> 4) << 24);   // -A B^T, N = 32
constexpr unsigned kT2ColALo = 240;   // TMEM columns 240..255: -A_lo of tile 0
constexpr unsigned kT2Idesc1T = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(kT2SJ >> 3) << 17) | ((128u >> 4) << 24);                   // A (negated already) from TMEM, N = 32
constexpr unsigned kT2Idesc2Hi = (1u << 4) | (2u << 7) | (2u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);                         // N = 32
constexpr unsigned kT2Idesc2Lo = (1u << 4) | (2u << 7) | (2u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);                         // N = 16

// The transposed image of GEMM 2 (the other arrays come from image_tc_kernel).  One thread per (partner quad, row n).
__global__ void __launch_bounds__(256) image_t2_kernel(RowDev dv, T2Image im) {
  if (__ldcg(&dv.state->stop)) return;
  const size_t x = (size_t)blockIdx.x * 256 + threadIdx.x;           // quad * 32 + n
  const size_t quad = x >> 5;
  const int n = (int)(x & 31);
  if (quad >= dv.cap_rows / 4) return;
  float4 hi = make_float4(0.f, 0.f, 0.f, 0.f), lo = hi;
  if (n < 16) {
    const float* r = im.a.rows32 + quad * 4 * 16 + n;                // rows32[partner][n], partners quad * 4 .. + 3
    const float v0 = r[0], v1 = r[16], v2 = r[32], v3 = r[48];
    hi = make_float4(tf32_round(v0), tf32_round(v1), tf32_round(v2), tf32_round(v3));
    lo = make_float4(v0 - hi.x, v1 - hi.y, v2 - hi.z, v3 - hi.w);
    reinterpret_cast<float4*>(im.ylo)[quad * 16 + n] = lo;
  } else if (n == 16) {
    hi = make_float4(1.f, 1.f, 1.f, 1.f);
  }
  reinterpret_cast<float4*>(im.yhi)[quad * 32 + n] = hi;
}

template <int H>
__global__ void __maxnreg__(80) repulse_tc2_kernel(RowDev dv, T2Image im, int cur, int cpi) {
  extern __shared__ __align__(128) unsigned char tc_smem[];
  constexpr int Dp = Row<H>::kStride;
  (void)cur;
  if (__ldcg(&dv.state->stop)) return;
  if (dv.adaptive && !form_is_tensor(dv)) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned sm0 = smem_u32(tc_smem);
  const unsigned bar_a_full = sm0 + T2Smem::kBars;
  auto bar_full = [&](int s) { return sm0 + T2Smem::kBars + 8u * (1 + s); };
  auto bar_empty = [&](int s) { return sm0 + T2Smem::kBars + 8u * (1 + kT2Stages + s); };
  auto bar_x = [&](int kind, int b) { return sm0 + T2Smem::kBars + 8u * (1 + 2 * kT2Stages + 2 * kind + b); };   // 0 tfull 1 wfull
  const unsigned bar_d2full = bar_x(2, 0), bar_d2empty = bar_x(2, 1), bar_a_tmem = bar_x(3, 0), bar_item = bar_x(3, 1);
  const unsigned bar_a_free = sm0 + T2Smem::kBars + 8u * (1 + 2 * kT2Stages + 8);
  unsigned* tmem_ptr_s = reinterpret_cast<unsigned*>(tc_smem + T2Smem::kTmemPtr);

  for (int s = 0; s < kT2Stages; ++s)
    for (int x = tid; x < kT2SJ * 4; x += kT2Threads)
      reinterpret_cast<float*>(tc_smem + T2Smem::kStage0 + s * T2Smem::kStageBytes + T2Smem::kBHi + 5 * kT2SJ * 16)[x] = 0.f;
  if (tid == 0) {
    mbar_init(bar_a_full, 1);
    mbar_init(bar_a_free, 1);
    for (int s = 0; s < kT2Stages; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 9); }   // 8 consumer warps + the commit of GEMM 2
    for (int b = 0; b < 2; ++b) { mbar_init(bar_x(0, b), 1); mbar_init(bar_x(1, b), 8); }
    mbar_init(bar_d2full, 1); mbar_init(bar_d2empty, 8); mbar_init(bar_a_tmem, 8); mbar_init(bar_item, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem0 = *tmem_ptr_s;
  auto col_s = [&](int b, int m) { return (unsigned)(b * 64 + m * 32); };           // S / w of buffer b, tile m
  auto col_d = [&](int m) { return (unsigned)(128 + m * 32); };                     // D2 of tile m
  auto col_a = [&](int m) { return (unsigned)(192 + m * 24); };                     // -A_hi of tile m: 16 coordinates, (h_hi, h_lo, 1, 1), 4 zeros

  const int tiles = dv.rows / kTcRows;
  const int groups = (dv.chunks + cpi - 1) / cpi;
  const long long items = (long long)tiles * groups;
  auto chunk_stages = [&](int c) { return (min(kChunk, dv.n - c * kChunk) + kT2SJ - 1) / kT2SJ; };

  // Work items are handed out by an atomic counter (the sums of an item do not depend on who computes it): CTAs that start
  // late or share their SM with a CTA of the spring walk (it runs under the pass) simply take fewer.  The copy warp
  // draws the CTA's next item and publishes it in a two-entry ring in shared memory (bar_item, one phase per item); it
  // publishes item k + 1 only after the consumers have started item k (bar_a_tmem), so no waiter can miss a phase.
  volatile int* item_ring = reinterpret_cast<volatile int*>(tc_smem + T2Smem::kTmemPtr) + 2;
  struct Cursor { long long item; int c, c_hi, s; size_t r0; bool valid; unsigned seq; };
  auto open_item = [&](Cursor& cu) {
    cu.valid = cu.item < items;
    if (!cu.valid) return;
    const int tile = (int)(cu.item / groups), grp = (int)(cu.item % groups);
    cu.c = grp * cpi; cu.c_hi = min(dv.chunks, cu.c + cpi); cu.s = 0;
    cu.r0 = (size_t)dv.row0 + (size_t)tile * kTcRows;
  };
  auto advance = [&](Cursor& cu) {
    if (++cu.s < chunk_stages(cu.c)) return;
    cu.s = 0;
    if (++cu.c < cu.c_hi) return;
    cu.valid = false;                 // the caller draws / takes the next item
  };
  auto draw_item = [&](Cursor& cu) {  // copy warp (converged)
    if (cu.seq > 0) mbar_wait(bar_a_tmem, (cu.seq - 1) & 1);
    // The MMA warp takes item k + 1 before it issues the last GEMM 2 of item k, which the consumers need before they can
    // start item k + 1 - so from item 2 on it cannot miss a phase of bar_item either.  Only its very first take has no
    // such anchor (the consumers write the rows' image of item 0 without it, and an item of <= 4 stages is loaded without
    // it): item 1 is published only after the GEMM 1s of item 0 (tests/tc2_protocol_model.py finds the hang without this).
    if (cu.seq == 1) mbar_wait(bar_a_free, 0);
    int id = 0;
    if (lane == 0) id = (int)atomicAdd(&dv.counters[2], 1u);
    id = __shfl_sync(0xffffffffu, id, 0);
    if (lane == 0) { item_ring[cu.seq & 1] = id; mbar_arrive(bar_item); }
    __syncwarp();
    ++cu.seq;
    cu.item = id;
    open_item(cu);
  };
  auto take_item = [&](Cursor& cu) {  // MMA warp (its leading cursor), consumer warps
    mbar_wait(bar_item, cu.seq & 1);
    cu.item = item_ring[cu.seq & 1];
    ++cu.seq;
    open_item(cu);
  };

  if (warp == 9) {
    // =========================== copy warp: shared-memory stages and the A tile of every item ===========================
    Cursor ld;
    ld.seq = 0;
    draw_item(ld);
    unsigned load_g = 0, item_g = 0;
    while (ld.valid) {
      if (ld.s == 0 && ld.c % cpi == 0) {
        // a new item: its A tile replaces the one the GEMM 1 of the item before read; the MMA warp commits a_free after the
        // last of them (this warp is at most one item boundary ahead of it: the phase waited for is the current one)
        if (item_g > 0) mbar_wait(bar_a_free, (item_g - 1) & 1);
        ++item_g;
        if (elect_one()) {
          mbar_expect_tx(bar_a_full, T2Smem::kATx);
          for (int c = 0; c < 4; ++c)      // the remainders of tile 1 (rows 128..255 of the item)
            bulk_g2s(sm0 + T2Smem::kALo1 + c * 128 * 16, im.a.xlo + ((size_t)c * dv.cap_rows + ld.r0 + 128) * 4, 128 * 16, bar_a_full);
        }
        __syncwarp();
      }
      const int s = load_g % kT2Stages;
      mbar_wait(bar_empty(s), ((load_g / kT2Stages) & 1) ^ 1);
      if (elect_one()) {
        const size_t j0 = (size_t)ld.c * kChunk + (size_t)ld.s * kT2SJ;
        const unsigned stg = sm0 + T2Smem::kStage0 + s * T2Smem::kStageBytes;
        mbar_expect_tx(bar_full(s), T2Smem::kStageTx);
        for (int c = 0; c < 4; ++c) {
          bulk_g2s(stg + T2Smem::kBHi + c * kT2SJ * 16, im.a.xhi + ((size_t)c * dv.cap_rows + j0) * 4, kT2SJ * 16, bar_full(s));
          bulk_g2s(stg + T2Smem::kBLo + c * kT2SJ * 16, im.a.xlo + ((size_t)c * dv.cap_rows + j0) * 4, kT2SJ * 16, bar_full(s));
        }
        bulk_g2s(stg + T2Smem::kBHi + 4 * kT2SJ * 16, im.a.aug_b + j0 * 4, kT2SJ * 16, bar_full(s));
        bulk_g2s(stg + T2Smem::kYHi, im.yhi + (j0 / 4) * 32 * 4, 8 * 32 * 16, bar_full(s));
        if (kT2LoPass) bulk_g2s(stg + T2Smem::kYLo, im.ylo + (j0 / 4) * 16 * 4, 8 * 16 * 16, bar_full(s));
        bulk_g2s(stg + T2Smem::kRows32, im.a.rows32 + j0 * 16, kT2SJ * 64, bar_full(s));
      }
      __syncwarp();
      ++load_g;
      advance(ld);
      if (!ld.valid) draw_item(ld);
    }
  } else if (warp == 8) {
    // =========================== MMA warp: GEMM 1 of stage g + 1, then GEMM 2 of stage g ===========================
    Cursor g1, g2;
    g1.seq = g2.seq = 0;
    int taken[2];                     // the leading cursor is at most one item ahead of the trailing one
    take_item(g1);
    taken[0] = (int)g1.item;
    g2.item = g1.item; g2.seq = 1;
    open_item(g2);
    unsigned g1_g = 0, g2_g = 0, a_uses = 0, chunk_g = 0;
    auto gemm1 = [&]() {
      if (g1.s == 0 && g1.c % cpi == 0) { mbar_wait(bar_a_full, a_uses & 1); mbar_wait(bar_a_tmem, a_uses & 1); ++a_uses; }
      const int s = g1_g % kT2Stages, b = g1_g & 1;
      mbar_wait(bar_full(s), (g1_g / kT2Stages) & 1);
      // buffer b: its last reader, GEMM 2 of stage g1_g - 2, was issued before this instruction (the tensor pipe runs in order)
      tc_fence_after();
      if (elect_one()) {
        const unsigned stg = sm0 + T2Smem::kStage0 + s * T2Smem::kStageBytes;
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          const unsigned d = tmem0 + col_s(b, m);
          const unsigned a_t = tmem0 + col_a(m), a_lo = sm0 + T2Smem::kALo1;
          const unsigned b_hi = stg + T2Smem::kBHi, b_lo = stg + T2Smem::kBLo;
          constexpr unsigned kLboA = 128 * 16, kLboB = kT2SJ * 16;
#pragma unroll
          for (int k = 0; k < 3; ++k)      // (-A_hi) B_hi^T, A from tensor memory (stored negated: no negate flag)
            tc_mma_tf32_ts(d, a_t + k * 8, tc_desc(b_hi + k * 2 * kLboB, kLboB, 128), kT2Idesc1T, k > 0);
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            tc_mma_tf32_ts(d, a_t + k * 8, tc_desc(b_lo + k * 2 * kLboB, kLboB, 128), kT2Idesc1T, 1);
            if (m == 0) tc_mma_tf32_ts(d, tmem0 + kT2ColALo + k * 8, tc_desc(b_hi + k * 2 * kLboB, kLboB, 128), kT2Idesc1T, 1);   // the last 16 columns
            else tc_mma_tf32(d, tc_desc(a_lo + k * 2 * kLboA, kLboA, 128), tc_desc(b_hi + k * 2 * kLboB, kLboB, 128), kT2Idesc1, 1);
          }
        }
        tc_commit(bar_x(0, b));
        if (g1.s + 1 == chunk_stages(g1.c) && g1.c + 1 == g1.c_hi) tc_commit(bar_a_free);   // the item's last GEMM 1
      }
      __syncwarp();
      ++g1_g;
      advance(g1);
      if (!g1.valid) { take_item(g1); taken[(g1.seq - 1) & 1] = (int)g1.item; }
    };
    auto gemm2 = [&]() {
      const int s = g2_g % kT2Stages, b = g2_g & 1;
      const bool first = g2.s == 0, last = g2.s + 1 == chunk_stages(g2.c);
      mbar_wait(bar_x(1, b), (g2_g >> 1) & 1);                       // the weights of the stage are in TMEM
      if (first) mbar_wait(bar_d2empty, (chunk_g & 1) ^ 1);          // the sums of the chunk before have been read
      tc_fence_after();
      if (elect_one()) {
        const unsigned stg = sm0 + T2Smem::kStage0 + s * T2Smem::kStageBytes;
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          const unsigned d = tmem0 + col_d(m), a = tmem0 + col_s(b, m);
#pragma unroll
          for (int k = 0; k < 4; ++k) {                                // 8 partners (two quads) per MMA
            // Y planes: per partner quad [32 rows][16 B] (hi) / [16 rows][16 B] (lo): LBO = next quad, SBO = 8 rows
            tc_mma_tf32_ts(d, a + k * 8, tc_desc(stg + T2Smem::kYHi + k * 2 * 512, 512, 128), kT2Idesc2Hi, !(first && k == 0));
            if (kT2LoPass) tc_mma_tf32_ts(d, a + k * 8, tc_desc(stg + T2Smem::kYLo + k * 2 * 256, 256, 128), kT2Idesc2Lo, 1);
          }
        }
        tc_commit(bar_empty(s));                                       // the stage's shared memory (and w buffer b) are free
        if (last) tc_commit(bar_d2full);
      }
      __syncwarp();
      if (last) ++chunk_g;
      ++g2_g;
      advance(g2);
      if (!g2.valid) { g2.item = taken[g2.seq & 1]; ++g2.seq; open_item(g2); }
    };
    if (g1.valid) gemm1();
    while (g2.valid) {
      // distances of the next stage while the consumers work on this one - except across an item boundary: the rows' image
      // of the next item is written to tensor memory by the consumers, who first need this item's last GEMM 2
      const bool boundary = g1.valid && g1.s == 0 && g1.c % cpi == 0;
      if (g1.valid && !boundary) gemm1();
      gemm2();
      if (boundary) gemm1();
    }
  } else {
    const int quad = warp & 3, half = warp >> 2;
    const unsigned lane_sel = (unsigned)(quad * 32) << 16;
    const bool series = dv.adaptive ? (__ldcg(&dv.counters[6]) == 2u) : (dv.series != 0);   // warp-uniform, fixed for the launch
    unsigned g = 0, chunk_g = 0, item_g = 0;
    Cursor cs;
    cs.seq = 0;
    for (;;) {
      take_item(cs);
      if (!cs.valid) break;
      const long long item = cs.item;
      const int tile = (int)(item / groups), grp = (int)(item % groups);
      const int c_lo = grp * cpi, c_hi = min(dv.chunks, c_lo + cpi);
      const int lrow[2] = {tile * kTcRows + quad * 32 + lane, tile * kTcRows + 128 + quad * 32 + lane};
      {
        // ---- the rows' image into tensor memory: warp (quad, half) writes rows quad * 32 .. + 31 of tile `half` ----
        if (item_g > 0) mbar_wait(bar_a_free, (item_g - 1) & 1);      // the GEMM 1s of the item before have read theirs
        ++item_g;
        tc_fence_after();
        const size_t grow = (size_t)dv.row0 + (size_t)(half ? lrow[1] : lrow[0]);
        const float4* xh = reinterpret_cast<const float4*>(im.a.xhi);
        const unsigned t_a = tmem0 + lane_sel + col_a(half);
#pragma unroll
        for (int cg = 0; cg < 2; ++cg) {
          const float4 u0 = __ldg(xh + (size_t)(2 * cg) * dv.cap_rows + grow), u1 = __ldg(xh + (size_t)(2 * cg + 1) * dv.cap_rows + grow);
          const unsigned v[8] = {__float_as_uint(-u0.x), __float_as_uint(-u0.y), __float_as_uint(-u0.z), __float_as_uint(-u0.w),
                                 __float_as_uint(-u1.x), __float_as_uint(-u1.y), __float_as_uint(-u1.z), __float_as_uint(-u1.w)};
          tc_st8(t_a + cg * 8, v);
        }
        {
          const float4 ag = __ldg(reinterpret_cast<const float4*>(im.a.aug_a) + grow);      // (-h_hi, -h_lo, -1, -1)
          const unsigned v[8] = {__float_as_uint(-ag.x), __float_as_uint(-ag.y), __float_as_uint(-ag.z), __float_as_uint(-ag.w), 0u, 0u, 0u, 0u};
          tc_st8(t_a + 16, v);
        }
        if (half == 0) {          // the remainders of tile 0 fill the last 16 columns (tile 1's stay in shared memory)
          const float4* xl = reinterpret_cast<const float4*>(im.a.xlo);
#pragma unroll
          for (int cg = 0; cg < 2; ++cg) {
            const float4 u0 = __ldg(xl + (size_t)(2 * cg) * dv.cap_rows + grow), u1 = __ldg(xl + (size_t)(2 * cg + 1) * dv.cap_rows + grow);
            const unsigned v[8] = {__float_as_uint(-u0.x), __float_as_uint(-u0.y), __float_as_uint(-u0.z), __float_as_uint(-u0.w),
                                   __float_as_uint(-u1.x), __float_as_uint(-u1.y), __float_as_uint(-u1.z), __float_as_uint(-u1.w)};
            tc_st8(tmem0 + lane_sel + kT2ColALo + cg * 8, v);
          }
        }
        tc_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_a_tmem);
      }
      float thr[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        thr[r] = -3.01e-3f * __ldg(im.a.aug_a + (size_t)(dv.row0 + lrow[r]) * 4);
        if (series) thr[r] = fmaxf(thr[r], kT2SeriesS);
      }
      for (int c = c_lo; c < c_hi; ++c, ++chunk_g) {
        float facc[32];
        bool fixed = false;
#pragma unroll
        for (int k = 0; k < 32; ++k) facc[k] = 0.f;
        const int nst = chunk_stages(c);
        for (int st = 0; st < nst; ++st, ++g) {
          const int s = g % kT2Stages, b = g & 1;
          mbar_wait(bar_full(s), (g / kT2Stages) & 1);
          mbar_wait(bar_x(0, b), (g >> 1) & 1);
          tc_fence_after();
          const float* __restrict__ q_s = reinterpret_cast<const float*>(tc_smem + T2Smem::kStage0 + s * T2Smem::kStageBytes + T2Smem::kRows32) + half * 16 * 16;
          const unsigned t_base = tmem0 + lane_sel + col_s(b, 0) + (unsigned)(half * 16);    // this warp's 16 partners of the stage, tile 0
#pragma unroll 1
          for (int bt = 0; bt < 2; ++bt) {
            unsigned s0[8], s1[8];
            tc_ld8(t_base + bt * 8, s0);
            tc_ld8(t_base + 32 + bt * 8, s1);
            tc_wait_ld();
            // w = (d + 0.01)^-3 with d = sqrt(2 S); a near pair gets -0: it adds nothing in GEMM 2 and is told apart from a
            // weight that underflowed to +0.  Near pairs are rare: one minimum per row and batch finds out whether there is
            // any (a compare and a select per pair would cost a fifth of the loop), the marking itself is out of the way.
            float m0 = __uint_as_float(s0[0]), m1 = __uint_as_float(s1[0]);
#pragma unroll
            for (int jj = 1; jj < 8; ++jj) { m0 = fminf(m0, __uint_as_float(s0[jj])); m1 = fminf(m1, __uint_as_float(s1[jj])); }
            const bool flag = (m0 < thr[0]) | (m1 < thr[1]);
            unsigned near_mask = 0u;
            if (flag) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj)
                near_mask |= (__uint_as_float(s0[jj]) < thr[0] ? (1u << jj) : 0u) | (__uint_as_float(s1[jj]) < thr[1] ? (256u << jj) : 0u);
            }
            if (series) {
              // one special-function instruction per pair: q = S^-1/2 = sqrt(2) / d, e = 0.01 / d <= 0.1 (closer pairs are
              // near pairs in this form), w = d^-3 (1 + e)^-3 = q^3 2^-1.5 p(e), p the cubic that interpolates (1 + e)^-3 at
              // the Chebyshev nodes of [0, 0.1]: 1.0e-5 relative (the weight is rounded to TF32, 4.9e-4, right after)
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                  const float q = rsqrt_approx_ftz(fabsf(__uint_as_float(r == 0 ? s0[jj] : s1[jj])));
                  const float q2 = q * q;
                  float pl = fmaf(-9.3722616e-07f, q, 1.0345994e-4f);
                  pl = fmaf(pl, q, -7.492801e-3f);
                  pl = fmaf(pl, q, 0.35355023f);
                  const float w = (q2 * q) * pl;
                  if (r == 0) s0[jj] = __float_as_uint(w); else s1[jj] = __float_as_uint(w);
                }
              }
            } else {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                  const float rc = rcp_approx_ftz(fmaf(sqrt_approx(fabsf(__uint_as_float(r == 0 ? s0[jj] : s1[jj]))), 1.41421356f, 0.01f));
                  const float w = (rc * rc) * rc;
                  if (r == 0) s0[jj] = __float_as_uint(w); else s1[jj] = __float_as_uint(w);
                }
              }
            }
            if (flag) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
                if (near_mask & (1u << jj)) s0[jj] = 0x80000000u;
                if (near_mask & (256u << jj)) s1[jj] = 0x80000000u;
              }
            }
            tc_st8(t_base + bt * 8, s0);
            tc_st8(t_base + 32 + bt * 8, s1);
            if (__any_sync(0xffffffffu, flag)) {
              if (flag) {
                fixed = true;
                unsigned sv[16];
                // the distances were overwritten by the weights: a near pair is one whose weight is -0
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) { sv[jj] = s0[jj]; sv[8 + jj] = s1[jj]; }
#pragma unroll 1
                for (int x = 0; x < 16; ++x) {
                  const int r = x >> 3, jj = x & 7;
                  if (sv[x] == 0x80000000u)
                    near_fix<H>(im.a.rows32 + (size_t)(dv.row0 + (r ? lrow[1] : lrow[0])) * 16, q_s + (bt * 8 + jj) * 16, facc + r * 16);
                }
              }
            }
          }
          tc_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { mbar_arrive(bar_x(1, b)); mbar_arrive(bar_empty(s)); }
        }
        // ---- the chunk's sums: warps of half h read tile h ----
        mbar_wait(bar_d2full, chunk_g & 1);
        tc_fence_after();
        {
          unsigned dlo[8], dhi[8];
          const unsigned d_base = tmem0 + lane_sel + col_d(half);
          tc_ld8(d_base, dlo);
          tc_ld8(d_base + 8, dhi);
          const float Wsum = __uint_as_float(tc_ld1(d_base + 16));
          tc_wait_ld();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_d2empty);
          // facc of the OTHER tile's rows lives in the other half's threads: exchange through shared memory would cost a
          // barrier; instead every thread adds its own near sums to the tile it writes... it only has them for its own
          // (half-specific) partners.  So near sums are written as their own partial entry (see below).
          const int r = half;
          float2 xi[H], o[H];
          ld_point<H>(im.a.rows32 + (size_t)(dv.row0 + lrow[r]) * 16, xi);
#pragma unroll
          for (int k = 0; k < H; ++k) {
            const float ax = __uint_as_float(k < 4 ? dlo[2 * k] : dhi[2 * k - 8]), ay = __uint_as_float(k < 4 ? dlo[2 * k + 1] : dhi[2 * k - 7]);
            o[k] = make_float2(fmaf(-xi[k].x, Wsum, ax), fmaf(-xi[k].y, Wsum, ay));
          }
          st_point<H>(dv.rpart + ((size_t)(3 * c) * dv.rows + lrow[r]) * Dp, o);
        }
        // near-pair sums of this thread's partner half, both rows: partial entries 3 c + 1 + half (zeros when there were none)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          float2 o[H];
#pragma unroll
          for (int k = 0; k < H; ++k) o[k] = make_float2(0.f, 0.f);
          if (fixed) {
#pragma unroll 1
            for (int k = 0; k < H; ++k) o[k] = make_float2(facc[r * 16 + 2 * k], facc[r * 16 + 2 * k + 1]);
          }
          st_point<H>(dv.rpart + ((size_t)(3 * c + 1 + half) * dv.rows + lrow[r]) * Dp, o);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem0), "r"(256) : "memory");
  }
}
