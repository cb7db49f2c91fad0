// topolow_b200/csrc/plan.cu
//
// Host driver of the production (coloured) mode and the single-fit / plan part of the C ABI declared in
// include/topolow_b200.h (the many-fits entry is batch.cu).  Builds the device image of one fit (relabelled positions, masses,
// bucketed edge records), picks the schedule geometry, launches the persistent kernel in
// chunks of iterations and assembles the five results of
// optimize_layout_exact_cpp (src/optimization.cpp:375-381).
#include <algorithm>
#include <cstring>
#include <memory>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <random>
#include <thread>
#include <map>
#include <functional>
#include <tuple>
#include <string>
#include <vector>

#include "../../include/topolow_b200.h"
#include "edges.h"
#include "replay.h"
#include "plan.h"
#include "rowblock.h"

using namespace tl;

namespace tl {

void validate(const topolow_problem& pb, const topolow_params& pr) {
  if (pb.n < 2) throw BadArg("Need at least 2 points for embedding");
  if (pb.ndim < 1) throw BadArg("ndim must be a positive integer");
  if (pr.n_iter < 0) throw BadArg("mapping_max_iter must be a positive integer");
  if (!pb.initial_positions || !pb.degrees) throw BadArg("initial_positions and degrees are required");
  if (pb.n_edges > 0 && (!pb.edge_i || !pb.edge_j || !pb.edge_dist || !pb.edge_thresh))
    throw BadArg("edge arrays are required when n_edges > 0");
  if (pb.n_edges < 0 || pb.n_edges >= (1ll << 32)) throw BadArg("n_edges out of range");
}

// Fisher-Yates with splitmix64: identical on every host.
std::vector<int32_t> random_permutation(int64_t n, uint64_t seed) {
  std::vector<int32_t> p(n);
  for (int64_t i = 0; i < n; ++i) p[i] = (int32_t)i;
  uint64_t s = mix64(seed ^ 0x51ab5eedULL);
  for (int64_t i = n - 1; i > 0; --i) {
    s += 0x9e3779b97f4a7c15ULL;
    const uint64_t r = mix64(s) % (uint64_t)(i + 1);
    std::swap(p[i], p[r]);
  }
  return p;
}

// Points per lane.  More points per lane = more work per shuffle and more independent chains in a
// lane, but n / (64 P) warps must still fill the 592 sub-partitions of the chip: measured on B200 (ms per
// iteration, 32 / 64 / 96-point tiles) n = 20k: 3.7 / 3.9 / 5.3, n = 40k: 8.5 / 7.8 / 10.6,
// n = 60k: - / 12.0 / 15.1, n = 100k: 25.8 / 27.9 / 23.8.  Batches of fits run one CTA each with
// 64-point tiles (topolow_fit_batch).
int choose_tile_points(int64_t n, int requested) {
  if (requested == 32 || requested == 64 || requested == 96) return requested / 32;
  return n >= 80000 ? 3 : (n >= 30000 ? 2 : 1);
}

int geometry_wmax(int D, int precision, int P, int max_warps) {
  const size_t rs = precision == TOPOLOW_PREC_F64_EXACT ? sizeof(double) : sizeof(float);
  int wmax = tile_max_warps(precision == TOPOLOW_PREC_F64_EXACT ? 1 : 0, P);
  if (max_warps > 0) wmax = std::min(wmax, max_warps);
  while (wmax > 1 && tile_smem_bytes(D, wmax, rs, P) > 224 * 1024) --wmax;
  return wmax;
}

// (G, m, W, S) of a kind-0 job over T tiles.
void shape_full(Geometry& g, int T, int wmax, int ctas) {
  if (T <= 2 * wmax || ctas == 1) {
    // one CTA: no inter-CTA barrier at all
    g.G = 1;
    g.m = (T + 2 * wmax - 1) / (2 * wmax);
    if (g.m < 1) g.m = 1;
    g.W = std::max(1, (T + 2 * g.m - 1) / (2 * g.m));
  } else if (T < 2 * ctas * std::min(4, wmax)) {
    // latency-bound regime: 4 warps per CTA, as many CTAs as there is work
    g.W = std::min(4, wmax); g.m = 1;
    g.G = (T + 2 * g.W - 1) / (2 * g.W);
  } else {
    // every SM busy; among CTA counts close to that pick the one with the fewest sub-round units
    // (2 G m rounds x m W sub-rounds): it wastes the fewest tile slots on padding.
    long best = -1;
    for (int G = ctas; G >= std::max(1, (ctas * 7) / 8); --G) {
      const int m = (T + 2 * G * wmax - 1) / (2 * G * wmax);
      const int W = (T + 2 * G * m - 1) / (2 * G * m);
      const long units = 2L * G * m * m * W;
      if (best < 0 || units * 100 < best * 99) { best = units; g.G = G; g.m = m; g.W = W; }  // >1 % better only
    }
  }
  g.S = 2 * g.G * g.m;
}
// (G, m, W, S) of a kind-1 job: S/2 = G*m super-blocks of W tiles on each side.
void shape_bipartite(Geometry& g, int count, int wmax, int ctas) {
  g.G = std::max(1, std::min(ctas, count));
  g.m = 1;
  g.W = (count + g.G - 1) / g.G;
  if (g.W > wmax) {
    g.m = (count + g.G * wmax - 1) / (g.G * wmax);
    g.W = (count + g.G * g.m - 1) / (g.G * g.m);
  }
  g.S = 2 * g.G * g.m;
}

Geometry choose_geometry(int64_t n, int D, int precision, int sms, int max_ctas, uint64_t seed, int max_warps = 0,
                         int P = 2, int n_shards = 0) {
  Geometry g{};
  g.n = (int)n; g.D = D; g.seed = seed; g.P = P;
  const int kTile = 32 * P;
  g.T = (int)((n + kTile - 1) / kTile);
  if (n_shards > 1) g.T = ((g.T + 2 * n_shards - 1) / (2 * n_shards)) * (2 * n_shards);   // equal mega-blocks
  const int wmax = geometry_wmax(D, precision, P, max_warps);
  const int ctas = std::max(1, max_ctas > 0 ? std::min(max_ctas, sms) : sms);
  shape_full(g, g.T, wmax, ctas);
  g.kind = 0; g.t0 = 0; g.tc = g.T; g.y0 = 0; g.yc = 0; g.do_end = 1;
  return g;
}

int64_t enumerate_schedule(const Geometry& g, const std::vector<int32_t>& pos, int iter, int32_t* out,
                           int64_t cap_pairs) {
  int64_t np = 0;
  bool overflow = false;
  const int kP = g.P, kTile = 32 * g.P;
  auto emit = [&](int slot_a, int slot_b) {
    const int pa = pos[slot_a], pb = pos[slot_b];   // -1: phantom slot (padding of the last / extra tiles)
    if (pa < 0 || pb < 0) return;
    if (np >= cap_pairs) { overflow = true; return; }
    out[2 * np] = pa; out[2 * np + 1] = pb; ++np;
  };
  auto ring = [&](int tA, int tB) {
    if (tA < 0 || tB < 0) return;
    const RingParams rp = ring_params(g, iter, tA, tB);
    for (int i = 0; i < 32; ++i)
      for (int w = 0; w < kP; ++w)
        for (int a = 0; a < 32; ++a)
          for (int p0 = 0; p0 < kP; ++p0)
            emit(tA * kTile + a + 32 * p0, tB * kTile + ring_b(rp, a, i) + 32 * ((p0 + w) % kP));
  };
  auto intra = [&](int t) {
    if (t < 0) return;
    const XorParams xp = xor_params(g, iter, t);
    for (int a = 0; a < 32; ++a)
      for (int p0 = 0; p0 < kP; ++p0)
        for (int q0 = p0 + 1; q0 < kP; ++q0) emit(t * kTile + a + 32 * p0, t * kTile + a + 32 * q0);
    for (int i = 0; i < 31; ++i) {
      const int x = xor_at(xp, i);
      for (int w = 0; w < kP; ++w)
        for (int a = 0; a < 32; ++a) if (a < (a ^ x))
          for (int p0 = 0; p0 < kP; ++p0)
            emit(t * kTile + a + 32 * p0, t * kTile + (a ^ x) + 32 * ((w - p0 + kP) % kP));
    }
  };
  const int W = g.W;
  for (int r = 0; r < cross_rounds(g); ++r) {
    const int rr = round_at(g, iter, r);
    for (int q = 0; q < g.S / 2; ++q) {
      int X, Y;
      cross_task(g, rr, q, X, Y);
      const int rot = cross_rot(g, iter, X, Y);
      for (int v = 0; v < W; ++v)
        for (int w = 0; w < W; ++w)
          ring(tile_at(g, iter, X * W + w, 0), tile_at(g, iter, Y * W + (w + v + rot) % W, g.kind));
    }
  }
  for (int q = 0; q < (g.kind == 0 ? g.S / 2 : 0); ++q) {
    const int Mt = diag_subrounds(W), rot = diag_rot(g, iter, q);
    for (int u = 0; u < Mt; ++u)
      for (int w = 0; w < W; ++w) {
        int sb, ia, ib;
        if (diag_pair(W, u, rot, w, sb, ia, ib))
          ring(tile_at(g, iter, (2 * q + sb) * W + ia), tile_at(g, iter, (2 * q + sb) * W + ib));
      }
    for (int w = 0; w < W; ++w) intra(tile_at(g, iter, (2 * q) * W + w));
    for (int w = 0; w < W; ++w) intra(tile_at(g, iter, (2 * q + 1) * W + w));
  }
  return overflow ? -2 : np;
}

template <class real>
void upload_points(topolow_plan& pl, const topolow_problem& pb, real phantom_coord) {
  const size_t slots = (size_t)pl.geo.T * 32 * pl.geo.P;
  std::vector<real> hp(slots * pl.D, phantom_coord), hd(slots, (real)0);
  for (int64_t i = 0; i < pl.n; ++i) {
    const size_t s = pl.store->slot_of_point[i];
    for (int d = 0; d < pl.D; ++d) hp[s * pl.D + d] = (real)pb.initial_positions[(size_t)d * pl.n + i];
    hd[s] = (real)((double)pb.degrees[i] + 1.0);
  }
  pool_alloc(pl.pos, hp.size() * sizeof(real));
  pool_alloc(pl.best, hp.size() * sizeof(real));
  pool_alloc(pl.dp1, hd.size() * sizeof(real));
  pool_ready();
  TL_CUDA(cudaMemcpy(pl.pos, hp.data(), hp.size() * sizeof(real), cudaMemcpyHostToDevice));
  TL_CUDA(cudaMemcpy(pl.best, hp.data(), hp.size() * sizeof(real), cudaMemcpyHostToDevice));
  TL_CUDA(cudaMemcpy(pl.dp1, hd.data(), hd.size() * sizeof(real), cudaMemcpyHostToDevice));
}

// Host-side bucket build for small edge lists (stable counting sort by tile pair; inside a bucket the
// records are then ordered by (slot_lo, slot_hi) exactly as the device path orders them).
void upload_edges(EdgeStore& st, const topolow_problem& pb, int T, int P) {
  const uint32_t kTile = 32u * (uint32_t)P;
  const size_t nkeys = (size_t)T * T;
  const int64_t E = pb.n_edges;
  std::vector<uint32_t> off(nkeys + 1, 0);
  std::vector<EdgeRec> recs(E);
  std::vector<uint32_t> keys(E);
  for (int64_t e = 0; e < E; ++e) {
    const int64_t a = pb.edge_i[e], b = pb.edge_j[e];
    if (a < 0 || b < 0 || a >= pb.n || b >= pb.n || a == b) throw BadArg("edge index out of range");
    uint32_t sa = (uint32_t)st.slot_of_point[a], sb = (uint32_t)st.slot_of_point[b];
    if (sa > sb) std::swap(sa, sb);  // lower slot first => lower (or equal) tile first
    keys[e] = (sa / kTile) * (uint32_t)T + (sb / kTile);
    off[keys[e] + 1]++;
  }
  for (size_t k = 0; k < nkeys; ++k) off[k + 1] += off[k];
  std::vector<uint32_t> cur(off.begin(), off.end() - 1);
  for (int64_t e = 0; e < E; ++e) {
    uint32_t sa = (uint32_t)st.slot_of_point[pb.edge_i[e]], sb = (uint32_t)st.slot_of_point[pb.edge_j[e]];
    if (sa > sb) std::swap(sa, sb);
    const int t = pb.edge_thresh[e];
    EdgeRec r;
    r.target = pb.edge_dist[e];
    r.slot_lo = sa;
    r.slot_hi_type = sb | ((uint32_t)(t == 0 ? 0 : (t == 1 ? 1 : 2)) << 30);   // src/optimization.cpp:237-243
    recs[cur[keys[e]]++] = r;
  }
  for (size_t k = 0; k < nkeys; ++k)
    if (off[k + 1] - off[k] > 1)
      std::sort(recs.begin() + off[k], recs.begin() + off[k + 1], [](const EdgeRec& x, const EdgeRec& y) {
        return x.slot_lo != y.slot_lo ? x.slot_lo < y.slot_lo
                                      : (x.slot_hi_type & 0x3fffffffu) < (y.slot_hi_type & 0x3fffffffu);
      });
  pool_alloc(st.edges, recs.size() * sizeof(EdgeRec));
  pool_alloc(st.bucket_off, off.size() * sizeof(uint32_t));
  pool_ready();
  if (!recs.empty()) TL_CUDA(cudaMemcpy(st.edges, recs.data(), recs.size() * sizeof(EdgeRec), cudaMemcpyHostToDevice));
  TL_CUDA(cudaMemcpy(st.bucket_off, off.data(), off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
}

// Relabelling + bucketed records of one edge list for tiles of 32 P points.  The relabelling is a
// fixed pseudo-random permutation of the points (it only has to decorrelate the caller's row order
// from the tiles; the per-fit randomness of the schedule comes from the seed-keyed hashes of
// schedule.h), so every fit of the same edge list can use the same store.
constexpr uint64_t kLayoutSeed = 0x746f706f6c6f77ULL;
std::shared_ptr<EdgeStore> make_store(const topolow_problem& pb, int T, int P, int device) {
  TL_CUDA(cudaSetDevice(device));
  keep_pool_memory(device);
  auto st = std::make_shared<EdgeStore>();
  st->device = device;
  st->slot_of_point = random_permutation(pb.n, kLayoutSeed);
  st->point_of_slot.assign((size_t)T * 32 * P, -1);
  for (int64_t i = 0; i < pb.n; ++i) st->point_of_slot[st->slot_of_point[i]] = (int32_t)i;
  if (pb.n_edges >= (1 << 21)) {
    StreamGuard stream;
    build_buckets(pb, st->slot_of_point, T, 32 * P, stream, &st->edges, &st->bucket_off);
  } else {
    upload_edges(*st, pb, T, P);   // small lists: a host counting sort beats a dozen device allocations
  }
  return st;
}

// shared: records + relabelling built for this edge list by the caller; shared_flag: two mapped host
// words of a block the caller owns (a batch allocates one block for all its plans).
std::unique_ptr<topolow_plan> make_plan(const topolow_problem& pb, const topolow_params& pr,
                                        std::shared_ptr<EdgeStore> shared, int* shared_flag) {
  validate(pb, pr);
  if (pb.ndim > kMaxDim) throw BadArg("ndim > 16 is not built into libtopolow_b200 (coloured mode); the row-block mode takes ndim <= 32, the replay mode any ndim");
  if (pb.n > 1000000) throw BadArg("n > 1,000,000 is not supported (bucket table is T x T)");
  if (pr.n_shards < 0 || pr.n_shards > 64) throw BadArg("n_shards must be in 0..64");
  auto pl = std::make_unique<topolow_plan>();
  pl->device = pr.device;
  TL_CUDA(cudaSetDevice(pr.device));
  keep_pool_memory(pr.device);
  int sms = 0;
  TL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, pr.device));
  pl->precision = pr.precision;
  pl->n = pb.n; pl->E = pb.n_edges; pl->D = pb.ndim;
  pl->prm = FitParams{pr.n_iter, pr.k0, pr.cooling_rate, pr.c_repulsion, pr.relative_epsilon,
                      pr.convergence_window, pr.convergence_check_freq};
  pl->n_shards = pr.n_shards > 1 ? pr.n_shards : 0;
  const int P = (pl->n_shards && pr.tile_points == 0) ? 1 : choose_tile_points(pb.n, pr.tile_points);
  pl->geo = choose_geometry(pb.n, pb.ndim, pr.precision, sms, pr.max_ctas, pr.seed, pr.max_warps, P, pl->n_shards);
  pl->wmax = geometry_wmax(pb.ndim, pr.precision, P, pr.max_warps);
  pl->ctas = std::max(1, pr.max_ctas > 0 ? std::min(pr.max_ctas, sms) : sms);
  const Geometry& g = pl->geo;
  if (g.G > 1) {
    const int fit = pr.precision == TOPOLOW_PREC_F64_EXACT ? max_coresident_f64(g.D, g.W, g.P) : max_coresident_f32(g.D, g.W, g.P);
    if (fit < g.G) throw BadArg("schedule does not fit the device (co-resident CTAs)");
  }
  pl->smem = tile_smem_bytes(g.D, g.W, pr.precision == TOPOLOW_PREC_F64_EXACT ? 8 : 4, g.P);

  PhaseTimer pt(nullptr);
  pt.mark("plan: geometry");
  // relabelling of points into slots (phantom slots pad the last tile) + bucketed edge records
  pl->store = shared ? shared : make_store(pb, g.T, g.P, pr.device);
  if ((int64_t)pl->store->slot_of_point.size() != pb.n || pl->store->point_of_slot.size() != (size_t)g.T * 32 * g.P)
    throw BadArg("shared edge store does not match the problem");
  pt.mark("plan: edges");
  if (pr.precision == TOPOLOW_PREC_F64_EXACT) upload_points<double>(*pl, pb, kPhantomCoordF64);
  else upload_points<float>(*pl, pb, kPhantomCoordF32);
  TL_CUDA(cudaStreamCreate(&pl->stream));
  pt.mark("plan: points");

  FitState st; state_init(st, pl->prm);
  // barrier: [0], [1] grid barrier; from word 32 on one round counter per super-block of any job geometry (S <= 2T + 2)
  const size_t barrier_words = 32 + 2 * (size_t)g.T + 64;
  const int ntr = std::max(pr.n_iter, 1);
  pool_alloc(pl->state, sizeof(FitState));
  pool_alloc(pl->partials, sizeof(double) * 4 * 1024);   // any job geometry: G <= SM count
  pool_alloc(pl->barrier, barrier_words * sizeof(unsigned));
  pool_alloc(pl->trace, sizeof(double) * ntr);
  pool_ready();
  TL_CUDA(cudaMemcpy(pl->state, &st, sizeof st, cudaMemcpyHostToDevice));
  TL_CUDA(cudaMemset(pl->partials, 0, sizeof(double) * 4 * 1024));
  TL_CUDA(cudaMemset(pl->barrier, 0, barrier_words * sizeof(unsigned)));
  std::vector<double> nanv(ntr, NAN);
  TL_CUDA(cudaMemcpy(pl->trace, nanv.data(), sizeof(double) * ntr, cudaMemcpyHostToDevice));
  if (pb.n_holdout > 0) {   // hold-out cells, relabelled to slots, wait on the device for the end of the fit
    if (!pb.holdout_i || !pb.holdout_j || !pb.holdout_truth) throw BadArg("hold-out arrays missing");
    std::vector<int32_t> si(pb.n_holdout), sj(pb.n_holdout);
    for (int64_t e = 0; e < pb.n_holdout; ++e) {
      const int64_t a = pb.holdout_i[e], b = pb.holdout_j[e];
      if (a < 0 || b < 0 || a >= pb.n || b >= pb.n) throw BadArg("hold-out index out of range");
      si[e] = pl->store->slot_of_point[a]; sj[e] = pl->store->slot_of_point[b];
    }
    pl->n_holdout = pb.n_holdout;
    pool_alloc(pl->hold_si, pb.n_holdout * sizeof(int32_t));
    pool_alloc(pl->hold_sj, pb.n_holdout * sizeof(int32_t));
    pool_alloc(pl->hold_truth, pb.n_holdout * sizeof(double));
    pool_ready();
    TL_CUDA(cudaMemcpy(pl->hold_si, si.data(), si.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    TL_CUDA(cudaMemcpy(pl->hold_sj, sj.data(), sj.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    TL_CUDA(cudaMemcpy(pl->hold_truth, pb.holdout_truth, pb.n_holdout * sizeof(double), cudaMemcpyHostToDevice));
  }
  if (shared_flag) { pl->h_flag = shared_flag; pl->owns_flag = false; }
  else TL_CUDA(cudaHostAlloc((void**)&pl->h_flag, 2 * sizeof(int), cudaHostAllocMapped));
  pl->h_flag[0] = 0; pl->h_flag[1] = 0;
  TL_CUDA(cudaHostGetDevicePointer((void**)&pl->d_flag, (void*)pl->h_flag, 0));
  TL_CUDA(cudaEventCreate(&pl->ev0));
  TL_CUDA(cudaEventCreate(&pl->ev1));

  // iterations per launch: aim at ~50 ms of device time, at most 50 iterations (the reference
  // polls for a user interrupt every 50 iterations, src/optimization.cpp:364)
  const double pairs = 0.5 * (double)pb.n * (double)(pb.n - 1);
  const double est_ms = pairs / 1.0e8 + 0.03;
  pl->chunk_iters = (int)std::max(1.0, std::min(50.0, 50.0 / est_ms));
  pt.mark("plan: state");
  if (const char* e = std::getenv("TOPOLOW_CHUNK_ITERS")) pl->chunk_iters = std::max(1, std::atoi(e));   // measurement aid
  return pl;
}

void launch_geo(topolow_plan& pl, const Geometry& geo, int n_iters, cudaStream_t stream) {
  if (pl.precision == TOPOLOW_PREC_F64_EXACT) launch_tile_f64(device_view<double>(pl), geo, pl.prm, n_iters, pl.d_flag, stream);
  else launch_tile_f32(device_view<float>(pl), geo, pl.prm, n_iters, pl.d_flag, stream);
  pl.launches++;
}
void launch_chunk(topolow_plan& pl, int n_iters, cudaStream_t stream) { launch_geo(pl, pl.geo, n_iters, stream); }

// Geometry of one job of a sharded iteration (see topolow_plan_run_job).
Geometry job_geometry(const topolow_plan& pl, int kind, int t0, int tc, int y0, int yc) {
  Geometry g = pl.geo;
  g.kind = kind; g.t0 = t0; g.tc = tc; g.y0 = y0; g.yc = yc; g.do_end = 0;
  if (kind == 0) shape_full(g, tc, pl.wmax, pl.ctas);
  else if (kind == 1) shape_bipartite(g, std::max(tc, yc), pl.wmax, pl.ctas);
  else g.do_end = 1;   // kind 2: the default geometry's CTAs run the end phase
  return g;
}
void check_job(const topolow_plan& pl, int kind, int t0, int tc, int y0, int yc) {
  const int T = pl.geo.T;
  if (kind < 0 || kind > 1 || t0 < 0 || tc < 1 || t0 + tc > T) throw BadArg("job tile range out of bounds");
  if (kind == 1 && (y0 < 0 || yc < 1 || y0 + yc > T || !(y0 >= t0 + tc || t0 >= y0 + yc)))
    throw BadArg("bipartite job needs two disjoint tile ranges");
}

// Runs up to n_iters iterations; returns device milliseconds.
double run_plan(topolow_plan& pl, int n_iters, cudaStream_t stream_in, topolow_interrupt_fn poll, void* user,
                bool* interrupted) {
  TL_CUDA(cudaSetDevice(pl.device));
  cudaStream_t s = stream_in ? stream_in : pl.stream;
  TL_CUDA(cudaEventRecord(pl.ev0, s));
  // never past n_iter (h_flag[1] = iterations done; every run_plan ends synchronised, so it is current here;
  // the kernel clamps as well)
  int left = std::min(n_iters, std::max(0, pl.prm.n_iter - (int)pl.h_flag[1]));
  while (left > 0) {
    if (pl.h_flag[0]) break;
    if (poll && poll(user)) { if (interrupted) *interrupted = true; break; }
    const int c = std::min(left, pl.chunk_iters);
    launch_chunk(pl, c, s);
    left -= c;
    if (poll) TL_CUDA(cudaStreamSynchronize(s));  // interruptible runs stay one chunk deep
  }
  TL_CUDA(cudaEventRecord(pl.ev1, s));
  TL_CUDA(cudaEventSynchronize(pl.ev1));
  float ms = 0.f;
  TL_CUDA(cudaEventElapsedTime(&ms, pl.ev0, pl.ev1));
  pl.total_ms += ms;
  return ms;
}

template <class real>
void download_best(const topolow_plan& pl, double* out) {
  const size_t slots = (size_t)pl.geo.T * 32 * pl.geo.P;
  std::vector<real> hp(slots * pl.D);
  TL_CUDA(cudaMemcpy(hp.data(), pl.best, hp.size() * sizeof(real), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < pl.n; ++i) {
    const size_t s = pl.store->slot_of_point[i];
    for (int d = 0; d < pl.D; ++d) out[(size_t)d * pl.n + i] = (double)hp[s * pl.D + d];
  }
}

void fill_result(topolow_plan& pl, topolow_result& res, bool interrupted) {
  TL_CUDA(cudaSetDevice(pl.device));
  FitState st;
  TL_CUDA(cudaMemcpy(&st, pl.state, sizeof st, cudaMemcpyDeviceToHost));
  if (res.positions) {
    if (pl.precision == TOPOLOW_PREC_F64_EXACT) download_best<double>(pl, res.positions);
    else download_best<float>(pl, res.positions);
  }
  res.converged = st.converged;
  res.iterations = st.best_iter;   // src/optimization.cpp:368-381: always the best snapshot
  res.final_mae = st.best_mae;
  res.final_k = st.best_k;
  res.iterations_run = st.iter;
  res.pair_updates = (int64_t)st.pair_updates;
  res.device_ms = pl.total_ms;
  res.holdout_sum_abs = 0.0; res.holdout_count = 0;
  if (pl.n_holdout > 0)
    holdout_resident(pl.best, pl.precision == TOPOLOW_PREC_F64_EXACT, pl.D, pl.n_holdout, pl.hold_si, pl.hold_sj,
                     pl.hold_truth, pl.stream, &res.holdout_sum_abs, &res.holdout_count);
  res.fail_iter = st.fail_iter;
  res.status = TOPOLOW_OK;
  res.message[0] = 0;
  if (st.status == 2) {
    res.status = TOPOLOW_ERR_NONFINITE;
    std::snprintf(res.message, sizeof res.message,
                  "Numerical instability at iteration %d. Reduce k0 or c_repulsion.", st.fail_iter);
  } else if (interrupted || st.status == kStatusStopped) {
    res.status = TOPOLOW_ERR_INTERRUPTED;
    std::snprintf(res.message, sizeof res.message, "interrupted");
  }
  if (res.trace_mae && pl.prm.n_iter > 0)
    TL_CUDA(cudaMemcpy(res.trace_mae, pl.trace, sizeof(double) * pl.prm.n_iter, cudaMemcpyDeviceToHost));
}

void print_trace(const topolow_params& pr, const double* trace, int iters_run) {
  // the reference's verbose lines (src/optimization.cpp:298-301), replayed from the device trace
  for (int it = 0; it < iters_run; ++it) {
    if (std::isnan(trace[it])) continue;
    if ((it + 1) % 10 == 0 || it == pr.n_iter - 1)
      std::fprintf(stderr, "Iter %d/%d, MAE=%g, k=%g\n", it + 1, pr.n_iter, trace[it],
                   pr.k0 * std::pow(1.0 - pr.cooling_rate, it + 1));
  }
}

int fit_impl(const topolow_problem* pb, const topolow_params* pr, topolow_result* res, topolow_interrupt_fn poll,
             void* user) {
  if (!pb || !pr || !res) return TOPOLOW_ERR_BAD_ARG;
  res->message[0] = 0;
  res->status = TOPOLOW_OK;
  res->holdout_sum_abs = 0.0; res->holdout_count = 0;
  try {
    if (pb->n < 2) {
      res->status = TOPOLOW_ERR_TOO_FEW_POINTS;
      set_msg(res->message, sizeof res->message, "Need at least 2 points for embedding");
      return res->status;
    }
    if (!res->positions) throw BadArg("result->positions must be caller-allocated");
    std::vector<double> tmp_trace;
    double* user_trace = res->trace_mae;
    if (pr->verbose && !res->trace_mae) { tmp_trace.assign(std::max(pr->n_iter, 1), NAN); res->trace_mae = tmp_trace.data(); }
    if (pr->mode == TOPOLOW_MODE_REPLAY) {
      validate(*pb, *pr);
      if (pb->n > replay_max_n()) throw BadArg("replay mode supports n <= 8192");
      if (pr->pair_order && pr->pairs_per_iter <= 0) throw BadArg("pairs_per_iter must be > 0 with pair_order");
      TL_CUDA(cudaSetDevice(pr->device));
      run_replay(*pb, *pr, *res, poll, user);
      if (res->status == TOPOLOW_OK && pb->n_holdout > 0 &&
          topolow_holdout_errors(res->positions, pb->n, pb->ndim, pb->n_holdout, pb->holdout_i, pb->holdout_j,
                                 pb->holdout_truth, &res->holdout_sum_abs, &res->holdout_count, pr->device) != TOPOLOW_OK)
        throw BadArg("hold-out cells out of range");
      if (res->status == TOPOLOW_ERR_NONFINITE)
        std::snprintf(res->message, sizeof res->message,
                      "Numerical instability at iteration %d. Reduce k0 or c_repulsion.", res->fail_iter);
    } else if (pr->mode == TOPOLOW_MODE_ROWBLOCK) {
      // host wall clock per phase under TOPOLOW_DEBUG (every phase ends synchronised)
      const bool dbg = std::getenv("TOPOLOW_DEBUG") != nullptr;
      auto t_last = std::chrono::steady_clock::now();
      auto lap = [&](const char* what) {
        if (!dbg) return;
        const auto now = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[topolow] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
      };
      {
        struct Holder { RowPlan* p; ~Holder() { row_destroy(p); } } h{row_create(*pb, *pr, 0, 1)};
        lap("fit: create");
        bool interrupted = false;
        row_run(*h.p, pr->n_iter, nullptr, poll, user, &interrupted);
        lap("fit: iterations");
        row_result(*h.p, *res, interrupted);
        lap("fit: result");
      }
      lap("fit: destroy");
    } else {
      auto pl = make_plan(*pb, *pr);
      bool interrupted = false;
      run_plan(*pl, pr->n_iter, nullptr, poll, user, &interrupted);
      fill_result(*pl, *res, interrupted);
    }
    if (pr->verbose && res->trace_mae) print_trace(*pr, res->trace_mae, res->iterations_run);
    res->trace_mae = user_trace;
    return res->status;
  } catch (const BadArg& e) {
    res->status = TOPOLOW_ERR_BAD_ARG;
    set_msg(res->message, sizeof res->message, e.what());
  } catch (const std::invalid_argument& e) {
    res->status = TOPOLOW_ERR_BAD_ARG;
    set_msg(res->message, sizeof res->message, e.what());
  } catch (const CudaError& e) {
    res->status = TOPOLOW_ERR_CUDA;
    set_msg(res->message, sizeof res->message, e.what());
    cudaGetLastError();
  } catch (const std::exception& e) {
    res->status = TOPOLOW_ERR_BAD_ARG;
    set_msg(res->message, sizeof res->message, e.what());
  }
  return res->status;
}

}  // namespace tl

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

const char* topolow_version(void) { return "topolow_b200 0.1 (sm_100a)"; }

void topolow_abi_sizes(int64_t out[3]) {
  out[0] = (int64_t)sizeof(topolow_problem); out[1] = (int64_t)sizeof(topolow_params); out[2] = (int64_t)sizeof(topolow_result);
}

int topolow_device_info(int32_t device, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* global_mem) {
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, device) != cudaSuccess) { cudaGetLastError(); return TOPOLOW_ERR_CUDA; }
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (global_mem) *global_mem = (int64_t)p.totalGlobalMem;
  return TOPOLOW_OK;
}

int topolow_fit(const topolow_problem* problem, const topolow_params* params, topolow_result* result) {
  return fit_impl(problem, params, result, nullptr, nullptr);
}

int topolow_fit_interruptible(const topolow_problem* problem, const topolow_params* params, topolow_result* result,
                              topolow_interrupt_fn poll, void* user) {
  return fit_impl(problem, params, result, poll, user);
}

int topolow_optimize_layout_exact(const double* initial_positions, int32_t n, int32_t ndim,
                                  const double* dissimilarity_matrix, const int32_t* threshold_matrix,
                                  const int32_t* degrees, const int32_t* edge_i, const int32_t* edge_j,
                                  const double* edge_dist, const int32_t* edge_thresh, int64_t n_edges, int32_t n_iter,
                                  double k0, double cooling_rate, double c_repulsion, double relative_epsilon,
                                  int32_t convergence_window, int32_t convergence_check_freq, int32_t verbose,
                                  double* positions_out, int32_t* converged_out, int32_t* iterations_out,
                                  double* final_mae_out, double* final_k_out, char* message, int32_t message_len) {
  // The dense matrices repeat the edge list (R/core.R:383-402 vs :429-436); when given, check it.
  if (dissimilarity_matrix) {
    for (int64_t e = 0; e < n_edges; ++e) {
      const int64_t a = std::min(edge_i[e], edge_j[e]), b = std::max(edge_i[e], edge_j[e]);
      if (a < 0 || b >= n) break;  // reported by validate()
      if (dissimilarity_matrix[a + b * (int64_t)n] != edge_dist[e] ||
          (threshold_matrix && threshold_matrix[a + b * (int64_t)n] != edge_thresh[e])) {
        set_msg(message, message_len, "dissimilarity_matrix / threshold_matrix disagree with the edge list");
        return TOPOLOW_ERR_BAD_ARG;
      }
    }
  }
  topolow_problem pb{};
  pb.n = n; pb.ndim = ndim; pb.n_edges = n_edges; pb.edge_i = edge_i; pb.edge_j = edge_j; pb.edge_dist = edge_dist;
  pb.edge_thresh = edge_thresh; pb.degrees = degrees; pb.initial_positions = initial_positions;
  topolow_params pr{};
  pr.n_iter = n_iter; pr.k0 = k0; pr.cooling_rate = cooling_rate; pr.c_repulsion = c_repulsion;
  pr.relative_epsilon = relative_epsilon; pr.convergence_window = convergence_window;
  pr.convergence_check_freq = convergence_check_freq; pr.verbose = verbose;
  topolow_result rs{};
  rs.positions = positions_out;
  const int rc = topolow_fit(&pb, &pr, &rs);
  if (converged_out) *converged_out = rs.converged;
  if (iterations_out) *iterations_out = rs.iterations;
  if (final_mae_out) *final_mae_out = rs.final_mae;
  if (final_k_out) *final_k_out = rs.final_k;
  set_msg(message, message_len, rs.message);
  return rc;
}

int topolow_plan_create(const topolow_problem* problem, const topolow_params* params, topolow_plan** plan_out,
                        char* message, int32_t message_len) {
  if (!problem || !params || !plan_out) return TOPOLOW_ERR_BAD_ARG;
  *plan_out = nullptr;
  try {
    if (params->mode != TOPOLOW_MODE_COLOURED) throw BadArg("plans exist for the coloured mode only");
    *plan_out = make_plan(*problem, *params).release();
    return TOPOLOW_OK;
  } catch (const CudaError& e) {
    set_msg(message, message_len, e.what()); cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  } catch (const std::exception& e) {
    set_msg(message, message_len, e.what());
    return problem->n < 2 ? TOPOLOW_ERR_TOO_FEW_POINTS : TOPOLOW_ERR_BAD_ARG;
  }
}

int topolow_plan_run(topolow_plan* plan, int32_t n_iters, void* stream, double* ms_out) {
  if (!plan) return TOPOLOW_ERR_BAD_ARG;
  try {
    const double ms = run_plan(*plan, n_iters, (cudaStream_t)stream, nullptr, nullptr, nullptr);
    if (ms_out) *ms_out = ms;
    return TOPOLOW_OK;
  } catch (const CudaError&) {
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  } catch (const std::exception&) {
    return TOPOLOW_ERR_BAD_ARG;
  }
}

int topolow_plan_result(topolow_plan* plan, topolow_result* result) {
  if (!plan || !result) return TOPOLOW_ERR_BAD_ARG;
  try {
    fill_result(*plan, *result, false);
    return result->status;
  } catch (const CudaError& e) {
    result->status = TOPOLOW_ERR_CUDA; set_msg(result->message, sizeof result->message, e.what()); cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  }
}

int topolow_plan_info(const topolow_plan* plan, int64_t* out, int32_t cap) {
  if (!plan || !out) return TOPOLOW_ERR_BAD_ARG;
  const Geometry& g = plan->geo;
  const int64_t v[13] = {g.T, g.S, g.W, g.G, g.m, g.S, (int64_t)plan->n * (plan->n - 1) / 2, (int64_t)plan->smem,
                         plan->chunk_iters, plan->launches, 32 * g.P,
                         plan->h_flag ? plan->h_flag[1] : 0, plan->h_flag ? plan->h_flag[0] : 0};   // as of the last finished launch
  for (int i = 0; i < cap && i < 13; ++i) out[i] = v[i];
  return TOPOLOW_OK;
}

// ---- sharded iteration: one job at a time ------------------------------------------------
int topolow_plan_run_job(topolow_plan* plan, int32_t kind, int32_t t0, int32_t tc, int32_t y0, int32_t yc, void* stream) {
  if (!plan) return TOPOLOW_ERR_BAD_ARG;
  try {
    TL_CUDA(cudaSetDevice(plan->device));
    check_job(*plan, kind, t0, tc, y0, yc);
    launch_geo(*plan, job_geometry(*plan, kind, t0, tc, y0, yc), 1, stream ? (cudaStream_t)stream : plan->stream);
    return TOPOLOW_OK;
  } catch (const CudaError&) {
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  } catch (const std::exception&) {
    return TOPOLOW_ERR_BAD_ARG;
  }
}

int topolow_plan_end_iteration(topolow_plan* plan, void* stream) {
  if (!plan) return TOPOLOW_ERR_BAD_ARG;
  try {
    TL_CUDA(cudaSetDevice(plan->device));
    launch_geo(*plan, job_geometry(*plan, 2, 0, 0, 0, 0), 1, stream ? (cudaStream_t)stream : plan->stream);
    return TOPOLOW_OK;
  } catch (const CudaError&) {
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  }
}

int topolow_plan_layout(const topolow_plan* plan, int64_t* out, int32_t cap) {
  if (!plan || !out) return TOPOLOW_ERR_BAD_ARG;
  const Geometry& g = plan->geo;
  const int64_t v[6] = {g.T, 32 * g.P, g.D, plan->precision == TOPOLOW_PREC_F64_EXACT ? 8 : 4, plan->n_shards,
                        (int64_t)g.T * 32 * g.P};
  for (int i = 0; i < cap && i < 6; ++i) out[i] = v[i];
  return TOPOLOW_OK;
}

void* topolow_plan_positions(topolow_plan* plan) { return plan ? plan->pos : nullptr; }

int64_t topolow_plan_enumerate_job(const topolow_plan* plan, int32_t iter, int32_t kind, int32_t t0, int32_t tc,
                                   int32_t y0, int32_t yc, int32_t* out, int64_t cap_pairs) {
  if (!plan || !out) return -1;
  try {
    check_job(*plan, kind, t0, tc, y0, yc);
    return enumerate_schedule(job_geometry(*plan, kind, t0, tc, y0, yc), plan->store->point_of_slot, iter, out, cap_pairs);
  } catch (const std::exception&) {
    return -1;
  }
}

void topolow_plan_destroy(topolow_plan* plan) { delete plan; }

// Host walk of the schedule the kernel executes (same functions, same loop nest).
int64_t topolow_plan_enumerate(const topolow_plan* plan, int32_t iter, int32_t* out, int64_t cap_pairs) {
  if (!plan || !out) return -1;
  return enumerate_schedule(plan->geo, plan->store->point_of_slot, iter, out, cap_pairs);
}

// The same walk without a device: geometry + relabelling are pure functions of
// (n, ndim, precision, sm_count, max_ctas, seed).  geometry_out (optional, 8 values) as in
// topolow_plan_info.
int64_t topolow_schedule_enumerate(int64_t n, int32_t ndim, int32_t precision, int32_t sm_count, int32_t max_ctas,
                                   uint64_t seed, int32_t iter, int32_t* out, int64_t cap_pairs,
                                   int64_t* geometry_out, int32_t tile_points) {
  if (n < 2 || ndim < 1 || ndim > kMaxDim || sm_count < 1) return -1;
  const Geometry g = choose_geometry(n, ndim, precision, sm_count, max_ctas, seed, 0, choose_tile_points(n, tile_points));
  if (geometry_out) {
    const int64_t v[8] = {g.T, g.S, g.W, g.G, g.m, g.S, n * (n - 1) / 2,
                          (int64_t)tile_smem_bytes(g.D, g.W, precision == TOPOLOW_PREC_F64_EXACT ? 8 : 4, g.P)};
    for (int i = 0; i < 8; ++i) geometry_out[i] = v[i];
  }
  if (!out) return 0;
  const std::vector<int32_t> sop = random_permutation(n, kLayoutSeed);   // as make_store()
  std::vector<int32_t> pos((size_t)g.T * 32 * g.P, -1);
  for (int64_t i = 0; i < n; ++i) pos[sop[i]] = (int32_t)i;
  return enumerate_schedule(g, pos, iter, out, cap_pairs);
}

}  // extern "C"
