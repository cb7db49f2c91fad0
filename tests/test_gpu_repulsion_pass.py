"""One repulsion pass of the row-block mode, isolated, against an FP64 reference of the same operation.

A map with no measured pairs (E = 0) runs one iteration: the spring walk leaves every row where it is, the one check
iteration finds MAE 0 and snapshots the positions after the pass, so

    P1_i - P0_i = -(c / 2) / (deg_i + 1) * sum_j (P0_j - P0_i) (|P0_j - P0_i| + 0.01)^-3

exactly as oracle/relaxed_oracle.cpp states step 1.  P0 is passed already FP32, so P1 - P0 is exact in FP64 and the only
difference between the kernel and the reference is the kernel's arithmetic (and the FP32 rounding of the stored P1).

Bars, per row i, with A_i = c / (2 (deg_i + 1)) sum_j w_ij |P_j - P_i| and r_i = (|d_gpu - d_ref| - 2^-23 |P1_i|)+ / A_i:
  tensor forms (11, weights by square root + reciprocal or by the series)   every r_i <= 1.5e-3, median <= 5e-4
      TF32 truncation of a weight <= 2^-10 (one-sided), S relative error <= 2.5e-4 -> w 4e-4, partners' TF32 rounding
  FP32 difference form (5)                                                  every r_i <= 1e-4, 99.9 % <= 1e-5
      w = 2^(-3 lg2(ds)) with sqrt / lg2 / ex2 approximate: <= 1.5e-6 relative; FP32 chunk sums over <= 2048 partners:
      <= 2048 x 2^-24 = 1.2e-4 if every rounding had the same sign, about sqrt(2048) x 2^-24 = 3e-6 as they come

Maps (`make_map`): points in the slots `structural_slots` names are planted in pairs 0.3 apart that carry >= 20 % of A_i
for both rows - a partner dropped at a stage, batch, half, chunk, tile or rank edge cannot hide among thousands of
similar terms.  `gemm`: the pairs sit within 3 of the centre, where they are far pairs of both GEMMs; `fixup`: 10..14
from it, where the tensor form re-does them from coordinate differences.  The rest of the map is a shell of radius
1.5 sqrt(n) .. 3 sqrt(n), mirrored point by point, and every coordinate is on a 2^-12 grid: the centroid is exactly 0
(1000 in the offset map), so the planted coordinates, on a coarser grid, are exact in TF32 and the partners' TF32
rounding - an error of 2^-11 |x_j| that the design accepts, not what these pairs test - leaves them alone.  The `gemm`
maps also carry an exact duplicate and pairs 0.05, 0.0999 and 0.1001 apart around the series form's near threshold.

Measured on one B200 1000 W, worst r_i / largest median r_i (maps of 100 rows or more) over the maps of this file:
  form 5         2.4e-5 at ndim 1, 5.4e-6 from ndim 2 on / 1.1e-6
  form 11        9.9e-4 / 2.6e-4
  form 11 series 9.9e-4 / 2.7e-4
The file ran in about 65 s there.
"""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, small_problem
from topolow_b200 import rowblock

sys.path.insert(0, os.path.join(ROOT, "tests"))
import tc2_arith_model as model  # noqa: E402

gpu = pytest.mark.gpu

GRID = 2.0 ** -12
FORMS = {"f32": {"TOPOLOW_REP_VARIANT": "5"},
         "tc": {"TOPOLOW_REP_VARIANT": "11", "TOPOLOW_TC_SERIES": "0"},
         "series": {"TOPOLOW_REP_VARIANT": "11", "TOPOLOW_TC_SERIES": "1"},
         "policy": {}}
BARS = {"f32": (1e-4, 0.999, 1e-5), "tc": (1.5e-3, 0.5, 5e-4), "series": (1.5e-3, 0.5, 5e-4)}   # (all rows, quantile, bar)
ENV = ("TOPOLOW_REP_VARIANT", "TOPOLOW_TC_SERIES", "TOPOLOW_ADAPTIVE", "TOPOLOW_OVERLAP", "TOPOLOW_NEAR_LIMIT")


# ------------------------------------------------------------------ maps ---------------------------------------------
def structural_slots(n):
    """Slots at the edges of the pass's work split: partner slots at the stage / batch / half edges of a full stage and
    of the last (ragged) stage, the chunk edges, the last slot, own rows at the quad / lane / tile edges of a 256-row
    item, and the first and last rows of every rank of a 2- and a 3-rank split."""
    s = {n - 1}
    for base in (32, (n - 1) // 32 * 32):
        s |= {base + k for k in (0, 7, 8, 15, 16, 31)}
    for c in range(1, (n - 1) // 2048 + 2):
        s |= {c * 2048 - 1, c * 2048, c * 2048 + 1}
    t = 256 if n > 511 else 0
    s |= {t + k for k in (0, 31, 32, 127, 128, 255)}
    tiles = (n + 255) // 256
    for g in (2, 3):
        if tiles >= g:
            for r in range(g):
                s |= {tiles * r // g * 256, tiles * (r + 1) // g * 256 - 1}
    return sorted(x for x in s if 0 <= x < n)


def _unit(rng, d):
    v = rng.normal(size=d)
    return v / np.linalg.norm(v)


def _q(v, grid):
    return np.round(np.asarray(v, np.float64) / grid) * grid


def _tf32_exact(v):
    return np.array_equal(model.tf32_rna(np.asarray(v, np.float32)), np.asarray(v, np.float32))


class Map:
    pass


def make_map(n, ndim, kind, seed, positions=None):
    """kind: 'gemm', 'fixup' (planted pairs, see the module's docstring), 'offset' ('gemm' + 1000 in every coordinate) or
    'clusters' (two tight clusters at +-50 along the first axis: nearly every pair inside a cluster is a near pair of the
    tensor form in every batch).  Returns a Map with P0 (FP32-exact, FP64), deg, c, planted = [(point, point)], rows
    that must be checked (`must`).  positions: use these (rounded to FP32) instead, with the same degrees."""
    rng = np.random.default_rng(seed)
    slot = rowblock.slot_order(n)
    point_of_slot = np.empty(n, np.int64)
    point_of_slot[slot] = np.arange(n)
    P = np.zeros((n, ndim))
    free = np.ones(n, bool)
    placed, planted, special = [], [], []

    def room(pts, sep):
        return all(np.linalg.norm(p - q) >= sep for p in pts for q in placed)

    def put(a, b, pa, pb):
        P[a], P[b] = pa, pb
        free[a] = free[b] = False
        placed.extend([pa, pb])

    if kind in ("gemm", "fixup", "offset"):
        slots = structural_slots(n)
        order = rng.permutation(len(slots))
        pts = [int(point_of_slot[slots[k]]) for k in order]
        near_centre = kind != "fixup"
        for a, b in zip(pts[0::2], pts[1::2]):
            for _ in range(400):
                r = rng.uniform(0.0, 3.0) if near_centre else rng.uniform(10.0, 14.0)
                grid = 2.0 ** -8 if near_centre else 2.0 ** -6
                pa = _q(_unit(rng, ndim) * r, grid)
                pb = _q(pa + 0.3 * _unit(rng, ndim), grid)
                if room([pa, pb], 1.0) and _tf32_exact(pa) and _tf32_exact(pb) and np.linalg.norm(pb) <= (3.2 if near_centre else 14.5):
                    put(a, b, pa, pb)
                    planted.append((a, b))
                    break
        if near_centre and n > 64:
            # around the series form's near threshold (d = 0.1: S = 0.005), and an exact duplicate
            for d in (0.05, 0.0999, 0.1001, 0.0):
                a, b = rng.choice(np.nonzero(free)[0], 2, replace=False)
                for _ in range(400):
                    pa = _q(_unit(rng, ndim) * rng.uniform(0.3, 1.5), 2.0 ** -6)
                    pb = pa.copy()
                    pb[rng.integers(ndim)] += _q(d, GRID)
                    if room([pa, pb], 0.6) and _tf32_exact(pa) and _tf32_exact(pb):
                        put(a, b, pa, pb)
                        special.append((a, b))
                        break
    rest = np.nonzero(free)[0]
    k = len(rest)
    s = P.sum(0)                                       # exact: every coordinate is on the grid
    if kind == "clusters":
        R0, half = 50.0, k // 2
        u = rng.normal(size=(half, ndim)) * (0.4 / np.sqrt(ndim))
        u *= np.minimum(1.0, 1.2 / np.maximum(np.linalg.norm(u, axis=1), 1e-12))[:, None]
        u[:, 0] += R0
        u = _q(u, GRID)
        cloud = np.vstack([u, -u] + ([np.zeros((1, ndim))] if k % 2 else []))
    else:
        R0 = 1.5 * np.sqrt(n) + 15.0
        m = max(k - 3, 0) // 2 if (k % 2) else max(k - 2, 0) // 2
        u = _q(np.array([_unit(rng, ndim) * rng.uniform(R0, 2 * R0) for _ in range(m)]).reshape(m, ndim), GRID)
        cloud = [u, -u]
        left = k - 2 * m
        if left >= 2:                                  # balance points: the whole map sums to exactly 0
            w1 = _q(_unit(rng, ndim) * R0, GRID)
            if left == 2:
                t = _q(-s / 2, GRID)
                cloud.append(np.stack([w1 + t, -w1 - s - t]))
            else:
                w2 = _q(-w1 / 2 + _unit(rng, ndim) * R0 / 2, GRID)
                cloud.append(np.stack([w1, w2, -w1 - w2 - s]))
        elif left == 1:
            cloud.append(-s[None, :])
        cloud = np.vstack(cloud)
    P[rest] = cloud[rng.permutation(k)] if k else cloud
    if kind == "offset":
        P += 1000.0
    if positions is not None:
        P = np.asarray(positions, np.float32).astype(np.float64)
        planted, special = [], []
    assert np.array_equal(P.astype(np.float32).astype(np.float64), P)
    mp = Map()
    mp.n, mp.ndim, mp.kind, mp.P0 = n, ndim, kind, P
    mp.deg = rng.integers(0, 51, n).astype(np.int32)
    mp.dp1 = mp.deg + 1.0
    mp.planted, mp.special = planted, special
    mp.must = np.unique(np.array([p for pr in planted + special for p in pr], dtype=np.int64))
    mp.rows = np.arange(n) if n <= 10000 else np.unique(np.r_[mp.must, rng.choice(n, 1500, replace=False)])
    F, A1 = reference_sums(P, mp.rows)
    d1 = np.linalg.norm(F, axis=1) / (2 * mp.dp1[mp.rows])
    scale = np.sqrt(((P - P.mean(0)) ** 2).sum(1).mean())
    mp.c = 0.05 * scale / np.median(d1)                # median |P1 - P0| = 5 % of the map's scale
    mp.F, mp.A1 = F, A1
    mp.d_ref = -(mp.c / (2 * mp.dp1[mp.rows]))[:, None] * F
    mp.A = mp.c / (2 * mp.dp1[mp.rows]) * A1
    return mp


def reference_sums(P, rows, budget=1 << 23):
    """FP64: (sum_j w_ij (P_j - P_i), sum_j w_ij |P_j - P_i|) for the rows `rows`, w = (|P_j - P_i| + 0.01)^-3."""
    n, d = P.shape
    bs = max(1, budget // (n * d))
    F, A = np.empty((len(rows), d)), np.empty(len(rows))
    for b in range(0, len(rows), bs):
        r = rows[b:b + bs]
        diff = P[None, :, :] - P[r, None, :]
        dist = np.sqrt((diff ** 2).sum(2))
        w = (dist + 0.01) ** -3
        F[b:b + len(r)] = np.einsum("rj,rjd->rd", w, diff)
        A[b:b + len(r)] = (w * dist).sum(1)
    return F, A


def planted_shares(mp):
    """Per planted pair, the share of A_i that the pair carries in each of its two rows."""
    pos = {int(p): k for k, p in enumerate(mp.rows)}
    out = []
    for a, b in mp.planted:
        dist = np.linalg.norm(mp.P0[a] - mp.P0[b])
        wd = dist / (dist + 0.01) ** 3
        out.append(min(wd / mp.A1[pos[a]], wd / mp.A1[pos[b]]))
    return np.array(out)


def ratios(mp, delta, P1=None):
    """r_i of the module's docstring for the rows mp.rows."""
    err = np.linalg.norm(delta - mp.d_ref, axis=1)
    if P1 is not None:
        err = np.maximum(err - 2.0 ** -23 * np.linalg.norm(P1, axis=1), 0.0)
    return err / mp.A


def assert_bars(r, form, what, ndim=16):
    """The bar on every row always; the quantile bar over 100 rows or more (with fewer, every row's sum is a planted pair
    or two, and the quantile is one pair's TF32 truncation, anywhere in [0, 2^-10]) and, for form 5, above ndim 1 (see
    test_fp32_form_sums_lose_the_far_partners_in_one_dimension)."""
    top, qu, qbar = BARS[form]
    worst, qv = float(r.max()), float(np.quantile(r, qu))
    print(f"{what} form {form}: worst r {worst:.3e}, median {float(np.median(r)):.3e}")
    assert worst <= top, f"{what} form {form}: worst r {worst:.3e} (row {int(r.argmax())})"
    if len(r) >= 100 and not (form == "f32" and ndim == 1):
        assert qv <= qbar, f"{what} form {form}: quantile {qu} {qv:.3e}"


# ------------------------------------------------------------------ running one pass -------------------------------------
def one_pass(monkeypatch, mp, form, n_ranks=1, **env):
    """(positions after one iteration, info of rank 0) - or, with n_ranks > 1, the positions of rank 0 and the last."""
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in {**FORMS[form], **env}.items():
        monkeypatch.setenv(k, v)
    e = np.zeros(0, np.int32)
    args = (mp.P0, mp.deg, e, e, np.zeros(0), e, 1, 1.0, 0.01, mp.c, 1e-4, 5, 1)
    if n_ranks == 1:
        sh = rowblock.Shard(*args, seed=5)
        try:
            sh.run(1)
            res, info = sh.result(), sh.info()
        finally:
            sh.close()
        assert res["iterations_run"] == 1 and res["status"] == 0
        return res["positions"], info
    ls = rowblock.LocalShards(*args, n_ranks=n_ranks, seed=5)
    try:
        ls.run(1)
        return [ls.result(rank=q)["positions"] for q in (0, n_ranks - 1)], ls.shards[0].info()
    finally:
        ls.close()


def check_form(monkeypatch, mp, form, what=""):
    pos, info = one_pass(monkeypatch, mp, form)
    P1 = pos[mp.rows]
    assert_bars(ratios(mp, P1 - mp.P0[mp.rows], P1), form, f"{what} n={mp.n} ndim={mp.ndim} {mp.kind}", mp.ndim)
    return pos, info


def check_all_forms(monkeypatch, mp, forms=("f32", "tc", "series", "policy")):
    got = {}
    for form in forms:
        if form == "policy":
            continue
        got[form] = check_form(monkeypatch, mp, form)[0]
    if "policy" in forms:
        pos, info = one_pass(monkeypatch, mp, "policy")
        if 5 <= mp.ndim <= 16:
            assert info["repulsion_form"] == 11 and info["tensor_form_iterations"] in (0, 1), info
            if info["tensor_form_iterations"] == 1:      # the probe picked one of the tensor forms for the iteration
                assert np.array_equal(pos, got["series"]) or np.array_equal(pos, got["tc"])
            else:
                assert np.array_equal(pos, got["f32"])
        else:
            assert info["repulsion_form"] == 5 and info["tensor_form_iterations"] == -1, info
            assert np.array_equal(pos, got["f32"])
    return got


# ------------------------------------------------------------------ CPU: the harness and its bars ---------------------------
def test_fp64_reference_is_the_first_iteration_of_the_relaxed_oracle():
    from oracle import cpu_oracle
    mp = make_map(700, 5, "gemm", 1)
    e = np.zeros(0, np.int32)
    want = cpu_oracle.relaxed_optimize_layout(mp.P0, mp.deg, e, e, np.zeros(0), e, 1, 1.0, 0.01, mp.c, 1e-4, 5, 1,
                                              seed=5, slot_of_point=rowblock.slot_order(mp.n))
    got = mp.P0 + mp.d_ref
    assert np.abs(want["positions"] - got).max() <= 1e-12 * np.abs(mp.P0).max()


@pytest.mark.parametrize("n,ndim,kind", [(2049, 1, "gemm"), (2049, 2, "fixup"), (2049, 3, "gemm"), (4129, 8, "fixup"),
                                         (2049, 15, "offset"), (3, 5, "gemm"), (33, 16, "fixup"), (257, 5, "gemm")])
def test_planted_maps_put_strong_pairs_at_the_structural_slots(n, ndim, kind):
    mp = make_map(n, ndim, kind, 7)
    slot = rowblock.slot_order(n)
    covered = {int(slot[p]) for pr in mp.planted for p in pr}
    want = set(structural_slots(n))
    if ndim >= 3:
        assert len(want - covered) <= 1, sorted(want - covered)     # an odd count leaves one slot to the shell
    assert len(mp.planted) >= min(3, len(want) // 2)
    assert planted_shares(mp).min() >= 0.2, planted_shares(mp)
    c = model.centre_of(mp.P0)
    assert np.all(c == (1000.0 if kind == "offset" else 0.0)) or n < 64
    x, _, _ = model.image(mp.P0)
    S, hh = model.distances(x, x)
    for a, b in mp.planted:
        for series in (False, True):
            near = model.near_mask(S[[a]], hh[[a]], series)[0, b]
            assert near == (kind == "fixup"), (a, b, series)
    med = np.median(np.linalg.norm(mp.d_ref, axis=1))
    scale = np.sqrt(((mp.P0 - mp.P0.mean(0)) ** 2).sum(1).mean())
    assert med == pytest.approx(0.05 * scale, rel=1e-9)


@pytest.mark.parametrize("n,ndim,kind", [(2049, 16, "gemm"), (2049, 16, "fixup"), (1500, 8, "clusters"), (2049, 15, "offset"),
                                         (2049, 1, "gemm"), (2049, 3, "fixup"), (1200, 5, "clusters")])
def test_emulated_tensor_pass_meets_the_tensor_bars(n, ndim, kind):
    mp = make_map(n, ndim, kind, 3)
    for series, form in ((False, "tc"), (True, "series")):
        F = model.tensor_pass(mp.P0, mp.rows, series=series)
        assert_bars(ratios(mp, -(mp.c / (2 * mp.dp1[mp.rows]))[:, None] * F), form, f"emulated {kind} ndim {ndim}")


@pytest.mark.parametrize("mutant", ["drop_last_stage_partner", "skip_near_fix", "no_plus_001", "pad_from_centre"])
def test_tensor_bars_catch_a_subtly_wrong_pass(mutant):
    """Each mutant of the emulated pass fails the tensor bars on the rows it affects, by a wide margin."""
    kind, ndim = {"skip_near_fix": ("fixup", 16), "pad_from_centre": ("offset", 15)}.get(mutant, ("gemm", 16))
    mp = make_map(2049, ndim, kind, 3)
    slot = rowblock.slot_order(mp.n)
    kw, rows = {}, mp.rows
    if mutant == "drop_last_stage_partner":
        last = int(np.nonzero(slot == mp.n - 1)[0][0])                # the point in the last slot: a ragged last stage
        mate = [b if a == last else a for a, b in mp.planted if last in (a, b)]
        assert mate, "the last slot is not planted"
        kw, rows = dict(drop=(last,)), np.array(mate)
    elif mutant == "skip_near_fix":
        kw, rows = dict(fix=False), mp.must
    elif mutant == "no_plus_001":
        kw, rows = dict(eps=0.0), [p for pr in mp.planted for p in pr]
    else:
        kw = dict(pad_from_centre=True)
    for series in (False, True):
        F = model.tensor_pass(mp.P0, mp.rows, series=series, **kw)
        r = ratios(mp, -(mp.c / (2 * mp.dp1[mp.rows]))[:, None] * F)
        hit = np.isin(mp.rows, rows)
        assert r[hit].min() > 20 * BARS["tc"][0], (mutant, series, r[hit].min())


def difference_form_sums(P):
    """sum_j w_ij (P_j - P_i) as repulse_kernel computes it for one chunk: FP32 differences and weights (correctly
    rounded here; the kernel's approximate sqrt / lg2 / ex2 add < 1e-6), accumulated in FP32 in slot order."""
    n = len(P)
    slot = rowblock.slot_order(n)
    point_of_slot = np.empty(n, np.int64)
    point_of_slot[slot] = np.arange(n)
    X = np.asarray(P, np.float32)[point_of_slot]
    f = np.float32
    acc = np.zeros_like(X)
    for j in range(n):
        dl = X[j][None, :] - X
        ds = np.sqrt((dl * dl).sum(1, dtype=f)) + f(0.01)
        acc = acc + dl * np.exp2(f(-3.0) * np.log2(ds))[:, None]
    return acc[slot].astype(np.float64)


def test_fp32_form_sums_lose_the_far_partners_in_one_dimension():
    """Why form 5's 99.9 % bar is not applied at ndim 1.  On a line, a row's FP32 running sum is set by its few close
    neighbours, and the thousand partners on the far side of the shell add terms below half an ulp of it, all of the same
    sign: they are lost together instead of rounding at random.  The FP32 form's own summation order reproduces the
    measured 2.2e-5 at 99.9 % (2.4e-5 worst) - within the every-row bound 2048 x 2^-24 = 1.2e-4 - and is an order of
    magnitude inside the 1e-5 bar from ndim 2 on."""
    for ndim, lo, hi in ((1, 1e-5, 1e-4), (2, 0.0, 1e-5)):
        mp = make_map(2049, ndim, "gemm", 100 + ndim)
        r = ratios(mp, -(mp.c / (2 * mp.dp1))[:, None] * difference_form_sums(mp.P0))
        assert lo < np.quantile(r, 0.999) <= hi and r.max() <= BARS["f32"][0], (ndim, np.quantile(r, 0.999), r.max())


# ------------------------------------------------------------------ GPU ---------------------------------------------------
@gpu
@pytest.mark.parametrize("ndim", range(1, 17))
def test_every_ndim_at_2049_points(monkeypatch, ndim):
    for kind in ("gemm", "fixup"):
        check_all_forms(monkeypatch, make_map(2049, ndim, kind, 100 + ndim))


@gpu
@pytest.mark.parametrize("ndim", [17, 20, 24, 32])
def test_wide_rows_at_2049_points(monkeypatch, ndim):
    check_all_forms(monkeypatch, make_map(2049, ndim, "gemm", 200 + ndim), forms=("f32", "policy"))


@gpu
@pytest.mark.parametrize("n", [2, 3, 33, 255, 256, 257, 2047, 2048, 2049, 4129])
def test_tile_stage_and_chunk_boundaries(monkeypatch, n):
    for ndim in (5, 8, 15, 16):
        for kind in ("gemm", "fixup"):
            check_all_forms(monkeypatch, make_map(n, ndim, kind, n + ndim))


@gpu
@pytest.mark.parametrize("kind,ndim", [("clusters", 8), ("clusters", 15), ("offset", 8), ("offset", 15)])
def test_two_clusters_and_an_offset_map(monkeypatch, kind, ndim):
    check_all_forms(monkeypatch, make_map(2049, ndim, kind, 300 + ndim))


@gpu
def test_cfg4_shape_groups_chunks_per_item(monkeypatch):
    """n = 100 000, ndim 16 (the benchmark's cfg4 shape): the tensor pass's items group several partner chunks (148 SMs:
    10 per item, the last group 9), the FP32 form's do not; sampled rows within the bars."""
    mp = make_map(100000, 16, "gemm", 4)
    _, info = check_form(monkeypatch, mp, "series")
    tiles = info["own_rows"] // 256
    assert info["repulsion_form"] == 11 and info["repulsion_items"] < tiles * info["partner_chunks"], info
    _, info = check_form(monkeypatch, mp, "f32")
    assert info["repulsion_items"] == tiles * info["partner_chunks"], info


@gpu
def test_policy_takes_the_series_tensor_form_on_a_spread_map_and_the_fp32_form_on_the_diagonal_start(monkeypatch):
    mp = make_map(2049, 16, "gemm", 9)
    series, _ = check_form(monkeypatch, mp, "series")
    pos, info = one_pass(monkeypatch, mp, "policy")
    assert info["tensor_form_iterations"] == 1 and np.array_equal(pos, series), info
    diag = make_map(2049, 16, "gemm", 9, positions=small_problem(2049, 16, 0.001, 9)[0])
    f32, _ = check_form(monkeypatch, diag, "f32")
    pos, info = one_pass(monkeypatch, diag, "policy")
    assert info["tensor_form_iterations"] == 0 and np.array_equal(pos, f32), info


@gpu
@pytest.mark.parametrize("form", ["series", "f32"])
def test_ranks_and_the_in_order_launch_give_the_same_bits(monkeypatch, form):
    """2 and 3 ranks in lock step (ranks 0 and last) and TOPOLOW_OVERLAP=0 give the bits of one rank with the overlapped
    launch: a chunk's partial sums do not depend on how the work is split or launched.  The planted rank-edge rows are
    within the bars."""
    mp = make_map(2049, 8, "gemm", 11)
    one, _ = check_form(monkeypatch, mp, form)
    for ranks in (2, 3):
        got, info = one_pass(monkeypatch, mp, form, n_ranks=ranks)
        assert info["n_ranks"] == ranks
        for q, pos in zip((0, ranks - 1), got):
            assert np.array_equal(pos, one), (ranks, q)
    pos, _ = one_pass(monkeypatch, mp, form, TOPOLOW_OVERLAP="0")
    assert np.array_equal(pos, one)
