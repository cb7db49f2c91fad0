"""CPU checks of tests/walk_model.py and of the bars of tests/test_gpu_spring_walk.py: the restatement is the first
iteration of the row-block oracle, the FP32 emulation of the walk stays well inside BETA, and every subtly wrong walk
(walk_model.MUTANTS) misses the bar by 10x or more on some row of the maps the GPU legs run."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from topolow_b200 import rowblock

sys.path.insert(0, os.path.join(ROOT, "tests"))
import walk_model as wm  # noqa: E402
import test_gpu_spring_walk as sw  # noqa: E402
from test_gpu_repulsion_pass import reference_sums  # noqa: E402

# the maps of test_gpu_spring_walk's legs (a): every ndim at 2049 points, three ndims at every size
WALK_MAPS = ([(2049, d, 10 + d) for d in sw.WALK_NDIMS]
             + [(n, d, n + d) for n in sw.WALK_NS for d in (3, 13, 24)])


@pytest.mark.parametrize("n,ndim,kind", [(5000, 3, "walk"), (2049, 8, "takeback"), (5000, 13, "sentinel")])
def test_walk_is_the_first_iteration_of_the_relaxed_oracle(n, ndim, kind):
    from oracle import cpu_oracle
    mp = sw.walk_map(n, ndim, {"walk": n + ndim, "takeback": 70 + ndim, "sentinel": 90 + n}[kind], kind)
    assert mp.recs.len.max() >= 2048
    ei, ej, ed, et = mp.edges
    want = cpu_oracle.relaxed_optimize_layout(mp.P0, mp.deg, ei, ej, ed, et, 1, sw.K0, 0.01, mp.c, 1e-4, 5, 1,
                                              seed=sw.SEED, slot_of_point=rowblock.slot_order(n))["positions"]
    F, _ = reference_sums(mp.P0, np.arange(n))
    R = -(mp.c / (2 * (mp.deg + 1.0)))[:, None] * F
    got = mp.ref["x"][mp.slot] + R
    scale = np.abs(mp.P0).max()
    assert np.abs(want - got).max() <= 1e-12 * scale, np.abs(want - got).max() / scale


@pytest.mark.parametrize("n,ndim,seed", WALK_MAPS)
def test_fp32_emulation_stays_within_a_quarter_of_beta(n, ndim, seed):
    mp = sw.walk_map(n, ndim, seed)
    em = wm.walk(mp.Ps, mp.dp1s, mp.recs, sw.K0, mp.c, sw.SEED, fp32=True)
    real = np.nonzero(mp.dp1s[:mp.recs.rows] > 0)[0]
    r = np.linalg.norm(em["x"][real] - mp.ref["x"][real], axis=1) / (mp.ref["B"][real] + sw.C_WALK)
    assert r.max() <= sw.BETA / 4, (r.max(), sw.BETA)


def _mutant_ratio(mp, mutant):
    recs = mp.recs
    if mutant in ("descending", "scatter_order"):
        recs = wm.build_records(mp.n, mp.edges, mp.slot, 0, mp.slots, mutant=mutant)
    got = wm.walk(mp.Ps, mp.dp1s, recs, sw.K0, mp.c, sw.SEED, mutant=mutant)
    P1s = mp.Ps.copy()
    P1s[:len(got["x"])] = got["x"]
    P1s[mp.slot] += mp.R
    return sw.ratios(mp, P1s)


@pytest.mark.parametrize("mutant", wm.MUTANTS)
def test_every_mutant_of_the_walk_fails_the_bar_by_10x(mutant):
    """The walk mutants on the hub map of legs (a) (n = 5000, three hub rows over 2048 records); the take-back is 1e-30
    of the coordinates there by design, so the take-back mutants run on a map of leg (c)."""
    if mutant in ("no_takeback", "takeback_from_x"):
        mp = sw.walk_map(2049, 8, 78, "takeback")
    else:
        mp = sw.walk_map(5000, 3, 5003)
    r = _mutant_ratio(mp, mutant)
    assert r.max() >= 10 * sw.BETA, (mutant, r.max())


def test_maps_reach_the_paths_the_legs_are_for():
    mp = sw.walk_map(5000, 3, 5003)
    ln = mp.recs.len
    assert {0, 1, 2047, 2048, 2049, 3000} <= set(ln.tolist())
    slices = ln[:mp.n // 32 * 32].reshape(-1, 32)
    assert any(len(set(s[mp.dp1s[32 * k:32 * k + 32] > 0].tolist())) > 8 for k, s in enumerate(slices))
    g = 2 * sw.K0 / (4 * (mp.deg + 1.0) + sw.K0)
    assert g.min() == pytest.approx(0.05) and g.max() == pytest.approx(0.5)
    # pairs listed twice with the same target, with another target and with another type
    ei, ej, ed, et = mp.edges
    key = np.minimum(ei, ej).astype(np.int64) * mp.n + np.maximum(ei, ej)
    _, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    twice = cnt[inv] > 1
    assert twice.sum() >= 20
    tb = sw.walk_map(2049, 8, 78, "takeback")
    for a, b, sat in tb.close:
        if not sat:
            d = np.linalg.norm(tb.P0[a] - tb.P0[b])
            share = d / (d + 0.01) ** 3 / tb.A1[[a, b]]
            assert share.min() >= 0.2, (a, b, share)
    # c = 1e-30: the repulsion and the take-back stay below 2^-60 of the coordinates, up to the 40k maps of legs (b)
    for m in (mp, sw.walk_map(2049, 1, 11)):
        assert 40000 * sw.W_MAX * 0.5 * sw.C_WALK <= 2.0 ** -60 * np.sqrt((m.P0 ** 2).sum(1).mean())
