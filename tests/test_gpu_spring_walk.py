"""The spring walk and the edge MAE of one row-block iteration, against an FP64 restatement (tests/walk_model.py).

Every leg runs one iteration with one check (n_iter = 1, convergence_check_freq = 1): the best state is P1, the position
after the iteration, and trace_mae[0] is the edge MAE on P1.

  (a) the walk alone: c_repulsion = 1e-30, so R_i and the take-back terms stay below 2^-60 of the coordinates and P1 is
      the walk's x.  Bar per row: |P1_i - x_i| <= BETA B_i (+ that bound on R_i), B_i the bar scale of walk_model.walk
      (sum over the visited records of |spring step| + |take-back| + g_i dist + |x|/16).
  (b) the production path of a map whose rank owns more than 2 x 148 row blocks of 128: the 4-deep ring, and under the
      two-GEMM form (ndim 5..16) a walk CTA that walks several row blocks.
  (c) take-back: a real c, the FP32 difference form (TOPOLOW_REP_VARIANT=5), spring pairs 0.05..0.3 apart whose take-back
      carries >= 20 % of the row's A_i.  Bar: BETA B_i + 1e-4 A_i (the difference form's bar of
      tests/test_gpu_repulsion_pass.py).
  (d) the edge MAE: trace_mae[0] against the FP64 MAE on the returned P1, |delta| <= 2^-21 sum (target + dist) / count;
      sentinel pairs whose |target - dist| is ~10^3 times the typical one at hub rows, rank, slice and duplicate edges
      (a record counted twice or not at all moves the MAE by ~10^3 / E); 1, 2 and 3 ranks give the same bits, and every
      rank's record totals are those of the restatement for its rows.

BETA = 2^-18, from the kernel's arithmetic: sqrt.approx / rcp.approx about 2^-22 relative, FP32 sums of dist2, one rounding
of x per step (|x|/16 in B_i carries 2^-24 |x| at 2^-20), targets already FP32: about 2^-21 per step of B_i.  The FP32
emulation of the walk (correctly rounded sqrt and reciprocal) stays below 2.6e-7 = BETA / 15 on the maps of (a)
(tests/test_spring_walk_model.py checks BETA / 4); every subtly wrong walk of walk_model.MUTANTS misses it by 200x or more.

Maps (`walk_map`): coordinates on a 2^-12 grid (exact in FP32); every slot of test_gpu_repulsion_pass.structural_slots
gets a record count from COUNTS (up to 3000 where n allows, different counts within a slice); the other rows get a
random sparse graph; pairs listed twice with the same target, with different targets and with different types; targets
dist0 U(0.5, 1.5), FP32-exact; thresholds resampled until every threshold record the walk visits, and every threshold
pair on P1, is at least 1e-3 (relative) from its target; degrees chosen so that g_i spans 0.05..0.5.

Measured on one B200 (1000 W), worst |P1_i - x_i| / B_i, by ring and H (= packed coordinate pairs, ndim 2H - 1..2H up to
ndim 16, 2H - 3..2H above):
  H               1       2       3       4       5       6       7       8       10      12      14      16
  8-deep ring   2.9e-7  3.0e-7  2.2e-7  1.9e-7  1.7e-7  1.7e-7  2.4e-7  1.7e-7  1.9e-7  2.2e-7  1.7e-7  2.0e-7
  4-deep ring   5.8e-7  3.6e-7  3.9e-7  2.8e-7  3.4e-7  3.4e-7  2.5e-7  2.9e-7  2.5e-7  2.4e-7  2.6e-7  2.2e-7
  (4-deep: the 40 000-point legs, one walk CTA per SM walking 2 or 3 row blocks at H 3..8; take-back legs 2.5e-7)
Edge MAE: |delta| at most 6.8e-4 of its bar; 1, 2 and 3 ranks and the overlapped launch gave the same bits.
The file's GPU legs ran in about 50 s there.
"""
import functools
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from topolow_b200 import rowblock

sys.path.insert(0, os.path.join(ROOT, "tests"))
import walk_model as wm  # noqa: E402
from test_gpu_repulsion_pass import ENV, reference_sums, structural_slots  # noqa: E402

gpu = pytest.mark.gpu

GRID = 2.0 ** -12
BETA = 2.0 ** -18          # 6.6 x the worst ratio measured (below), 4 x the FP32 emulation's worst
K0 = 4.0                  # g_i = 2 k / (4 (deg_i + 1) + k) = 2 / (deg_i + 2): deg 2..38 gives 0.5..0.05
C_WALK = 1e-30
SEED = 5
COUNTS = (0, 1, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 2047, 2048, 2049, 3000)
MARGIN = 1e-3
WALK_NDIMS = (1, 2, 3, 4, 5, 6, 8, 9, 11, 12, 13, 14, 15, 16, 17, 19, 21, 24, 26, 28, 29, 32)
WALK_NS = (2, 3, 31, 33, 257, 2049, 5000)
BIG_NDIMS = (2, 4, 6, 8, 10, 12, 14, 16, 20, 24, 28, 32)     # one per H = 1..8, 10, 12, 14, 16
# max over j of |P_j - P_i| / (|P_j - P_i| + 0.01)^3 (at 0.005): bounds every repulsion and take-back weight
W_MAX = 0.005 / 0.015 ** 3


def _q(v, grid=GRID):
    return np.round(np.asarray(v, np.float64) / grid) * grid


class WalkMap:
    pass


@functools.lru_cache(maxsize=None)
def walk_map(n, ndim, seed, kind="walk"):
    """kind 'walk' (c = 1e-30), 'takeback' (planted close spring and satisfied threshold pairs, a real c) or 'sentinel'
    ('walk' with the sentinel pairs of (d))."""
    rng = np.random.default_rng(seed)
    slot = rowblock.slot_order(n).astype(np.int64)
    pos = np.empty(n, np.int64)
    pos[slot] = np.arange(n)
    scale = 1.5 * np.sqrt(n) + 15.0
    P = _q(rng.normal(size=(n, ndim)) * scale / np.sqrt(ndim))
    deg = rng.integers(2, 39, n).astype(np.int32)
    struct = [int(pos[s]) for s in structural_slots(n)]
    is_struct = np.zeros(n, bool)
    is_struct[struct] = True
    free = np.nonzero(~is_struct)[0]
    ei, ej, et, close = [], [], [], []

    def add(a, b, t):
        ei.append(a), ej.append(b), et.append(t)

    types = np.array([0, 0, 0, 1, -1])
    if len(free) >= 2:                                   # the rest of the map: about 6 records per row
        m = 3 * len(free)
        a, b = rng.choice(free, m), rng.choice(free, m)
        for x, y in zip(a[a != b], b[a != b]):
            add(int(x), int(y), int(rng.choice(types)))
    if kind == "takeback":                               # close pairs of structural points, 0.05..0.3 apart
        order = rng.permutation(struct)
        for k, (a, b) in enumerate(zip(order[0::2], order[1::2])):
            u = rng.normal(size=ndim)
            P[b] = _q(P[a] + rng.uniform(0.05, 0.3) * u / np.linalg.norm(u), 2.0 ** -8)
            close.append((int(a), int(b), k % 2))        # 0: exact pair (a spring), 1: satisfied threshold
    counts = [c for c in COUNTS if c <= n - 1]
    counts = counts[-4:] + list(rng.permutation(counts[:-4]))   # the hubs first, then the rest in random order
    for k, p in enumerate(rng.permutation(struct)):
        c = counts[k % len(counts)]
        pool = free[free != p] if len(free[free != p]) else np.delete(np.arange(n), p)
        partners = rng.choice(pool, c, replace=c > len(pool))
        for q in partners:
            add(int(p), int(q), int(rng.choice(types)))
    ei, ej, et = np.array(ei, np.int64), np.array(ej, np.int64), np.array(et, np.int32)
    dist0 = np.linalg.norm(P[ei] - P[ej], axis=1)
    ed = np.maximum(dist0, 2.0 ** -8) * rng.uniform(0.5, 1.5, len(ei))
    # pairs listed twice: the same target, another target, another type
    cand = np.nonzero(~is_struct[ei] & ~is_struct[ej])[0]
    dup = rng.choice(cand, min(30, len(cand)), replace=False)
    mp_dups = np.arange(len(ei), len(ei) + len(dup))
    extra_d, extra_t = [], []
    for k, e in enumerate(dup):
        extra_d.append(ed[e] * (1.0 if k % 3 != 1 else rng.uniform(0.5, 1.5)))
        extra_t.append(et[e] if k % 3 != 2 else (1 if et[e] == 0 else 0))
    if len(dup):
        ei, ej = np.r_[ei, ei[dup]], np.r_[ej, ej[dup]]
        ed, et = np.r_[ed, extra_d], np.r_[et, np.array(extra_t, np.int32)]
    for a, b, sat in close:                              # the planted pairs' own edges
        d = np.linalg.norm(P[a] - P[b])
        ei, ej = np.r_[ei, a], np.r_[ej, b]
        ed = np.r_[ed, d * (rng.uniform(0.5, 1.5) if not sat else rng.uniform(0.5, 0.8))]
        et = np.r_[et, np.int32(1 if sat else 0)]        # '>' with target < dist: satisfied, keeps its repulsion
    sentinels = []
    if kind == "sentinel":
        typical = np.median(np.abs(ed - np.linalg.norm(P[ei] - P[ej], axis=1)))
        ss = structural_slots(n)
        rows = [int(pos[s]) for s in ss]                 # hubs, slice edges, rank edges of 2- and 3-rank splits
        for p in rows:
            inc = np.nonzero(((ei == p) | (ej == p)) & (et == 0))[0]
            if len(inc):
                sentinels.append(int(inc[0]))
        if len(mp_dups):
            sentinels.append(int(mp_dups[-1]))            # the second copy of a pair listed twice
        sentinels = np.unique(sentinels)
        ed[sentinels] = np.linalg.norm(P[ei[sentinels]] - P[ej[sentinels]], axis=1) + 1e3 * typical
        et[sentinels] = 0
    ed = ed.astype(np.float32).astype(np.float64)
    mp = WalkMap()
    mp.n, mp.ndim, mp.kind, mp.P0, mp.deg, mp.slot, mp.pos = n, ndim, kind, P, deg, slot, pos
    mp.slots = (n + 255) // 256 * 256
    mp.Ps = np.zeros((mp.slots, ndim))
    mp.Ps[slot] = P
    mp.dp1s = np.zeros(mp.slots)
    mp.dp1s[slot] = deg + 1.0
    mp.sentinels, mp.close = sentinels, close
    if kind == "takeback":
        F, A1 = reference_sums(P, np.arange(n))
        scale_p = np.sqrt(((P - P.mean(0)) ** 2).sum(1).mean())
        d1 = np.linalg.norm(F, axis=1) / (2 * (deg + 1.0))
        mp.c = 0.05 * scale_p / np.median(d1)
        mp.R = -(mp.c / (2 * (deg + 1.0)))[:, None] * F  # point order
        mp.A = mp.c / (2 * (deg + 1.0)) * A1
        mp.A1 = A1
    else:
        mp.c = C_WALK
        mp.R, mp.A = np.zeros_like(P), np.zeros(n)
    # the repulsion and take-back terms of c = 1e-30: n W_MAX c / 2 at most
    mp.r_bound = n * W_MAX * 0.5 * C_WALK if kind != "takeback" else 0.0
    for _ in range(30):
        mp.edges = (ei.astype(np.int32), ej.astype(np.int32), ed, et)
        mp.recs = wm.build_records(n, mp.edges, slot, 0, mp.slots)
        mp.ref = wm.walk(mp.Ps, mp.dp1s, mp.recs, K0, mp.c, SEED)
        P1 = mp.Ps.copy()
        P1[:len(mp.ref["x"])] = mp.ref["x"]
        P1[slot] += mp.R
        mp.P1s = P1
        d1 = np.linalg.norm(P1[slot[ei]] - P1[slot[ej]], axis=1)
        low_p1 = np.nonzero((et != 0) & (np.abs(d1 - ed) < MARGIN * ed))[0]
        low = np.union1d(mp.ref["low"], low_p1)
        if not len(low):
            break
        ed = ed.copy()
        ed[low] = (np.maximum(np.linalg.norm(P[ei[low]] - P[ej[low]], axis=1), 2.0 ** -8)
                   * rng.uniform(0.5, 1.5, len(low))).astype(np.float32).astype(np.float64)
    assert not len(low), f"{len(low)} threshold pairs within {MARGIN} of their target after resampling"
    assert mp.ref["margin"].min() >= MARGIN
    return mp


def ratios(mp, P1s, rows=None):
    """|P1_i - x_i - R_i| / (B_i + slack / BETA) per own slot with a point (slot order)."""
    rows = np.arange(mp.n) if rows is None else rows          # points
    s = mp.slot[rows]
    want = mp.ref["x"][s] + mp.R[rows]
    err = np.linalg.norm(P1s[s] - want, axis=1)
    slack = (mp.r_bound + 1e-4 * mp.A[rows]) / BETA
    return err / (mp.ref["B"][s] + slack + 1e-300)


def run(monkeypatch, mp, n_ranks=0, **env):
    """One iteration: Shard (n_ranks = 0: the production launch) or LocalShards (n_ranks >= 1, in lock step).
    Returns ([(positions in slot order, trace_mae[0]) per rank], [info per rank])."""
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ei, ej, ed, et = mp.edges
    args = (mp.P0, mp.deg, ei, ej, ed, et, 1, K0, 0.01, mp.c, 1e-4, 5, 1)
    out, infos = [], []

    def take(res):
        assert res["iterations_run"] == 1 and res["status"] == 0, res
        P1s = np.zeros_like(mp.Ps)
        P1s[mp.slot] = res["positions"]
        out.append((P1s, float(res["trace_mae"][0])))

    if n_ranks == 0:
        sh = rowblock.Shard(*args, seed=SEED)
        try:
            sh.run(1)
            take(sh.result(trace=True))
            infos.append(sh.info())
        finally:
            sh.close()
    else:
        ls = rowblock.LocalShards(*args, n_ranks=n_ranks, seed=SEED)
        try:
            ls.run(1)
            for q in range(n_ranks):
                take(ls.result(rank=q, trace=True))
                infos.append(ls.shards[q].info())
        finally:
            ls.close()
    return out, infos


def check_walk(mp, P1s, what):
    r = ratios(mp, P1s)
    print(f"{what}: worst |P1 - x| / B = {r.max():.3e} (beta {BETA:.3e})")
    assert r.max() <= BETA, f"{what}: worst ratio {r.max():.3e} at point {int(r.argmax())} > {BETA:.3e}"
    return float(r.max())


# ------------------------------------------------------------------ GPU ---------------------------------------------------
@gpu
@pytest.mark.parametrize("ndim", WALK_NDIMS)
def test_walk_alone_every_h(monkeypatch, ndim):
    mp = walk_map(2049, ndim, 10 + ndim)
    (res,), (info,) = run(monkeypatch, mp)
    assert info["walk_ring"] == 8, info
    check_walk(mp, res[0], f"n=2049 ndim={ndim} H={wm.row_width(ndim) // 2} ring 8")


@gpu
@pytest.mark.parametrize("n", WALK_NS)
def test_walk_alone_sizes_and_hubs(monkeypatch, n):
    for ndim in (3, 13, 24):
        mp = walk_map(n, ndim, n + ndim)
        if n == 5000:
            assert {2047, 2048, 2049, 3000} <= set(mp.recs.len.tolist())
        (res,), (info,) = run(monkeypatch, mp)
        assert info["walk_ring"] == 8, info
        check_walk(mp, res[0], f"n={n} ndim={ndim} ring 8")


@gpu
@pytest.mark.parametrize("ndim", BIG_NDIMS)
def test_walk_of_a_rank_with_many_row_blocks(monkeypatch, ndim):
    """40 000 points, one rank: 40 192 own rows = 314 row blocks > 2 x 148, so the walk takes the 4-deep ring; under the
    two-GEMM form (the policy's form for ndim 5..16) the walk runs one CTA per SM, each walking several row blocks."""
    mp = walk_map(40000, ndim, 40 + ndim)
    (res,), (info,) = run(monkeypatch, mp)
    assert info["own_rows"] == 40192 and info["walk_ring"] == 4, info
    if 5 <= ndim <= 16:
        assert info["repulsion_form"] == 11 and info["walk_ctas"] < info["own_rows"] // 128, info
    else:
        assert info["repulsion_form"] == 5 and info["walk_ctas"] == info["own_rows"] // 128, info
    assert info["spring_records"] == mp.recs.spring_records and info["mae_records"] == mp.recs.mae_records, info
    check_walk(mp, res[0], f"n=40000 ndim={ndim} H={wm.row_width(ndim) // 2} ring 4 walk_ctas {info['walk_ctas']}")


@gpu
@pytest.mark.parametrize("ndim", [3, 8, 16])
def test_take_back_of_close_spring_pairs(monkeypatch, ndim):
    mp = walk_map(2049, ndim, 70 + ndim, "takeback")
    (res,), (info,) = run(monkeypatch, mp, TOPOLOW_REP_VARIANT="5")
    assert info["repulsion_form"] == 5
    check_walk(mp, res[0], f"take-back n=2049 ndim={ndim}")


def _mae_check(mp, P1s, mae, what):
    s, cnt, scale, _ = wm.mae_terms(P1s, mp.recs)
    tol = 2.0 ** -21 * scale / cnt
    print(f"{what}: MAE {mae:.9e} vs FP64 {s / cnt:.9e}: |d| / tol = {abs(mae - s / cnt) / tol:.3e}")
    assert abs(mae - s / cnt) <= tol, (what, mae, s / cnt, tol)


@gpu
@pytest.mark.parametrize("n", [2049, 5000])
def test_edge_mae_and_records_over_ranks(monkeypatch, n):
    mp = walk_map(n, 7, 90 + n, "sentinel")
    assert len(mp.sentinels) >= 5
    (one,), (info1,) = run(monkeypatch, mp, n_ranks=1)
    _, _, _, mg = wm.mae_terms(one[0], mp.recs)
    assert mg >= MARGIN / 2, mg                      # no threshold on P1 is close enough for FP32 to decide otherwise
    _mae_check(mp, one[0], one[1], f"n={n} 1 rank")
    for ranks in (2, 3):
        got, infos = run(monkeypatch, mp, n_ranks=ranks)
        for q, ((P1s, mae), info) in enumerate(zip(got, infos)):
            assert np.array_equal(P1s, one[0]) and mae == one[1], (ranks, q)
            want = wm.build_records(n, mp.edges, mp.slot, info["row0"], info["own_rows"])
            assert (info["spring_records"], info["mae_records"]) == (want.spring_records, want.mae_records), (ranks, q, info)
    got, (info,) = run(monkeypatch, mp)                # the overlapped production launch gives the same bits
    assert np.array_equal(got[0][0], one[0]) and got[0][1] == one[1]


# ------------------------------------------------------------------ refused threshold codes ------------------------------
@pytest.mark.parametrize("code", [2, -2])
def test_threshold_codes_outside_minus_one_to_one_are_refused(code):
    """validate() runs before any device call, so this needs no GPU: the coloured and the row-block mode refuse the code."""
    from topolow_b200 import _lib
    rng = np.random.default_rng(0)
    init = rng.normal(size=(6, 2))
    deg = np.full(6, 2, np.int32)
    ei, ej = np.array([0, 1, 2], np.int32), np.array([1, 2, 3], np.int32)
    ed, et = np.array([1.0, 1.0, 1.0]), np.array([0, code, 1], np.int32)
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(init, deg, ei, ej, ed, et, 2, 4.0, 0.01, 0.02)
    assert e.value.status == _lib.ERR_BAD_ARG and "edge_thresh must be -1, 0 or 1" in str(e.value)
    with pytest.raises(_lib.TopolowError) as e:
        rowblock.Shard(init, deg, ei, ej, ed, et, 2, 4.0, 0.01, 0.02)
    assert e.value.status == _lib.ERR_BAD_ARG and "edge_thresh must be -1, 0 or 1" in str(e.value)
