"""GPU parity tests (run with -m gpu on the B200 box).  Everything goes through the C ABI
(topolow_b200._lib -> libtopolow_b200.so); the oracle is only the checker.

Bars:
  replay mode (FP64)              bit-exact positions / iterations / k vs the seeded CPU loop and vs the
                                  golden vectors produced by the reference's own source; MAE within 1e-12
  coloured mode, FP64 exact       bit-exact positions vs the CPU loop run on the enumerated pair order
  coloured mode, FP32 production  vs the FP64 run of the same order after a few iterations: 99 % of the coordinates
                                  within 2e-4 of the coordinate scale, all within 1e-3; statistical parity (MAE over 10 seeds) vs the reference's
                                  random-shuffle loop: |mean difference| <= max(2 x pooled SE, 2 % relative)
"""
import ctypes as C

import numpy as np
import pytest

from conftest import load_fixture, load_golden, random_r_matrix, small_problem
from oracle import cpu_oracle, r_glue
from tools import synth
from topolow_b200 import _lib, core, cv
from topolow_b200.sharded import ShardedMap

pytestmark = pytest.mark.gpu

GOLDENS = ["triangle", "small_thresholds", "small_sparse", "h3n2_ndim5", "hiv_ndim5"]


# ------------------------------------------------------------------ replay mode ----------------
@pytest.mark.parametrize("name", GOLDENS)
def test_replay_reproduces_reference_golden(name):
    z, args, seed = load_golden(name)
    got = _lib.fit(*args, mode=_lib.MODE_REPLAY, seed=seed)
    assert np.array_equal(got["positions"], z["positions"])          # bit for bit
    assert got["iterations"] == int(z["iterations"])
    assert got["converged"] == bool(z["converged"])
    assert got["final_k"] == float(z["final_k"])
    assert got["final_mae"] == pytest.approx(float(z["final_mae"]), rel=1e-12)


def test_replay_explicit_order_and_early_convergence():
    args = small_problem(70, 3, 0.3, 4)
    want = cpu_oracle.optimize_layout_exact(*args, 300, 5.0, 0.03, 0.02, 1e-3, 3, 2, seed=5, trace=True)
    got = _lib.fit(*args, 300, 5.0, 0.03, 0.02, 1e-3, 3, 2, mode=_lib.MODE_REPLAY, seed=5, trace=True)
    assert want["converged"] and want["iterations"] < 300           # exercises the early exit
    assert np.array_equal(got["positions"], want["positions"])
    assert (got["iterations"], got["converged"]) == (want["iterations"], want["converged"])
    np.testing.assert_allclose(got["trace_mae"][: got["iterations_run"]], want["trace_mae"][: got["iterations_run"]],
                               rtol=1e-12, equal_nan=True)
    order = cpu_oracle.pair_orders(70, 12, 9)
    w2 = cpu_oracle.optimize_layout_exact(*args, 12, 5.0, 0.03, 0.02, pair_order=order)
    g2 = _lib.fit(*args, 12, 5.0, 0.03, 0.02, mode=_lib.MODE_REPLAY, pair_order=order)
    assert np.array_equal(g2["positions"], w2["positions"])


def test_replay_positions_in_global_memory_path():
    # n * ndim * 8 bytes exceeds the shared-memory budget of the replay kernel: positions stay in L2
    args = small_problem(900, 24, 0.02, 77)
    want = cpu_oracle.optimize_layout_exact(*args, 3, 5.0, 0.01, 0.02, seed=11)
    got = _lib.fit(*args, 3, 5.0, 0.01, 0.02, mode=_lib.MODE_REPLAY, seed=11)
    assert np.array_equal(got["positions"], want["positions"])
    assert got["pair_updates"] == 3 * 900 * 899 // 2


# ------------------------------------------------------------------ coloured mode, exact ------
def _exact_case(args, iters, hp, seed, max_ctas=0, tile_points=0):
    plan = _lib.Plan(*args, iters, *hp, precision=_lib.PREC_F64_EXACT, seed=seed, max_ctas=max_ctas,
                     tile_points=tile_points)
    order = np.stack([plan.enumerate(it) for it in range(iters)])
    info = plan.info()
    plan.run(iters)
    got = plan.result()
    plan.close()
    want = cpu_oracle.optimize_layout_exact(*args, iters, *hp, pair_order=order)
    return got, want, info


@pytest.mark.parametrize("tile_points", [32, 64, 96])
@pytest.mark.parametrize("n,d,dens", [(3, 2, 1.0), (33, 2, 0.5), (100, 7, 0.15), (150, 3, 0.2), (260, 16, 0.05)])
def test_coloured_fp64_equals_cpu_loop_on_the_enumerated_order(n, d, dens, tile_points):
    args = small_problem(n, d, dens, n)
    got, want, info = _exact_case(args, 7, (5.0, 0.01, 0.02, 1e-4, 5, 3), seed=n, tile_points=tile_points)
    assert info["tile_points"] == tile_points
    assert np.array_equal(got["positions"], want["positions"])
    assert got["iterations"] == want["iterations"] and got["final_k"] == want["final_k"]
    assert got["final_mae"] == pytest.approx(want["final_mae"], rel=1e-12)
    assert got["pair_updates"] == 7 * n * (n - 1) // 2


@pytest.mark.parametrize("tile_points", [32, 64, 96])
def test_coloured_fp64_multi_cta_barrier_path(tile_points):
    # n = 1100 -> more tiles than one CTA holds -> several co-operating CTAs (grid barrier between rounds)
    args = small_problem(1100, 4, 0.03, 12)
    got, want, info = _exact_case(args, 3, (5.0, 0.01, 0.02, 1e-4, 5, 3), seed=2, tile_points=tile_points)
    assert info["ctas"] > 1
    assert np.array_equal(got["positions"], want["positions"])
    # and a forced multi-task-per-CTA geometry
    got, want, info = _exact_case(args, 2, (5.0, 0.01, 0.02, 1e-4, 5, 3), seed=3, max_ctas=2, tile_points=tile_points)
    assert info["tasks_per_cta"] >= 1 and info["ctas"] == 2
    assert np.array_equal(got["positions"], want["positions"])


@pytest.mark.parametrize("fixture,hp", [("h3n2", (14.76214, 0.03641074, 0.002943064)),
                                        ("hiv", (3.550036, 0.04130713, 0.0007038619))])
def test_coloured_fp64_on_bundled_data(fixture, hp):
    # BASELINE.json configs[0] / configs[1]: real titers incl. '<' / '>' thresholds, ndim = 5
    f = load_fixture(fixture)
    init = np.random.default_rng(1).normal(size=(int(f["n"]), 5))
    args = (init, f["degrees"], f["edge_i"], f["edge_j"], f["edge_dist"], f["edge_thresh"])
    got, want, _ = _exact_case(args, 10, (*hp, 1e-4, 5, 3), seed=4)
    assert np.array_equal(got["positions"], want["positions"])


def test_coloured_convergence_controller_matches():
    args = small_problem(90, 3, 0.3, 6, thresholds=False)
    hp = (5.0, 0.05, 0.02, 1e-2, 2, 2)
    got, want, _ = _exact_case(args, 120, hp, seed=1)
    assert want["converged"] and want["iterations"] < 120
    assert (got["converged"], got["iterations"]) == (want["converged"], want["iterations"])
    assert np.array_equal(got["positions"], want["positions"])


@pytest.mark.parametrize("world,tile_points,n", [(2, 32, 700), (4, 32, 1100), (2, 64, 900), (3, 96, 1300)])
def test_sharded_map_is_one_sequential_order(world, tile_points, n):
    """The multi-GPU schedule (mega-block tournament, bipartite + diagonal jobs) emulated on one GPU:
    exact FP64 equals the CPU loop on the enumerated order, bit for bit."""
    args = small_problem(n, 4, 0.04, 40 + n)
    hp = (5.0, 0.01, 0.02, 1e-4, 5, 3)
    sm = ShardedMap(*args, 4, *hp, world_size=world, precision=_lib.PREC_F64_EXACT, seed=5, tile_points=tile_points,
                    emulate=True)
    order = [sm.enumerate(it) for it in range(4)]
    P = n * (n - 1) // 2
    for o in order:                       # every pair exactly once per iteration
        key = np.minimum(o[:, 0], o[:, 1]).astype(np.int64) * n + np.maximum(o[:, 0], o[:, 1])
        assert len(o) == P and len(np.unique(key)) == P
    sm.step(4)
    got = sm.result()
    sm.close()
    want = cpu_oracle.optimize_layout_exact(*args, 4, *hp, pair_order=np.stack(order))
    assert np.array_equal(got["positions"], want["positions"])
    assert got["iterations"] == want["iterations"] and got["final_k"] == want["final_k"]
    assert got["final_mae"] == pytest.approx(want["final_mae"], rel=1e-12)


# ------------------------------------------------------------------ coloured mode, FP32 -------
@pytest.mark.parametrize("tile_points,f64_warps", [(32, 8), (64, 4), (96, 2)])
@pytest.mark.parametrize("n,d,dens", [(150, 3, 0.2), (300, 16, 0.05), (285, 5, 0.08), (1100, 5, 0.03)])
def test_fp32_tracks_fp64_on_the_same_order(n, d, dens, tile_points, f64_warps):
    args = small_problem(n, d, dens, 100 + n)
    hp = (5.0, 0.01, 0.02, 1e-4, 50, 3)
    a = _lib.fit(*args, 6, *hp, precision=_lib.PREC_F64_EXACT, seed=8, tile_points=tile_points)
    b = _lib.fit(*args, 6, *hp, precision=_lib.PREC_F32, seed=8, tile_points=tile_points,
                 max_warps=f64_warps)   # max_warps: the schedule the FP64 plan gets
    scale = max(np.abs(a["positions"]).max(), 1.0)
    err = np.abs(a["positions"] - b["positions"])
    # a close approach of two points (force ~ 1/(d + 0.01)^3) can amplify FP32 rounding for those points
    assert np.quantile(err, 0.99) <= 2e-4 * scale and err.max() <= 1e-3 * scale
    assert b["final_mae"] == pytest.approx(a["final_mae"], rel=1e-3)


def test_statistical_parity_with_the_random_shuffle_loop():
    """Production schedule + FP32 vs the reference's std::shuffle loop (oracle), 10 seeds, same inputs:
    the edge MAE at the best state and the in-sample mae of R/core.R:481 must agree within
    max(2 x SE of the difference, 2 %)."""
    n, d = 160, 3
    gpu, cpu = [], []
    for seed in range(10):
        args = small_problem(n, d, 0.15, 1000 + seed, thresholds=True)
        hp = (5.0, 0.01, 0.02, 1e-4, 5, 3)
        cpu.append(cpu_oracle.optimize_layout_exact(*args, 150, *hp, seed=seed)["final_mae"])
        gpu.append(_lib.fit(*args, 150, *hp, precision=_lib.PREC_F32, seed=seed)["final_mae"])
    gpu, cpu = np.array(gpu), np.array(cpu)
    diff = gpu.mean() - cpu.mean()
    se = np.sqrt(gpu.var(ddof=1) / 10 + cpu.var(ddof=1) / 10)
    assert abs(diff) <= max(2 * se, 0.02 * cpu.mean()), (gpu, cpu)


def test_heldout_mae_parity_with_the_random_shuffle_loop():
    """The north-star acceptance check: on the same training edges and initial positions the production
    mode reproduces the reference loop's HELD-OUT MAE (cells the fit never saw) and its distance-
    reconstruction error (all measured cells, train + held-out) - mean over 10 seeds within
    max(2 x SE of the difference, 3 %)."""
    n, d = 180, 3
    res = {"gpu": ([], []), "cpu": ([], [])}
    for seed in range(10):
        init, deg, ei, ej, ed, et = small_problem(n, d, 0.2, 2000 + seed, thresholds=False)
        rng = np.random.default_rng(seed)
        held = rng.random(len(ei)) < 0.1
        tr = ~held
        deg_tr = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
        train = (init, deg_tr, ei[tr], ej[tr], ed[tr], et[tr])
        hp = (5.0, 0.01, 0.02, 1e-4, 5, 3)
        g = _lib.fit(*train, 200, *hp, precision=_lib.PREC_F32, seed=seed, holdout=(ei[held], ej[held], ed[held]))
        c = cpu_oracle.optimize_layout_exact(*train, 200, *hp, seed=seed)
        for key, pos, hold_mae in (("gpu", g["positions"], g["holdout_sum_abs"] / g["holdout_count"]),
                                   ("cpu", c["positions"], None)):
            dist = np.linalg.norm(pos[ei] - pos[ej], axis=1)
            if hold_mae is None:
                hold_mae = np.abs(ed[held] - dist[held]).mean()
            else:
                assert hold_mae == pytest.approx(np.abs(ed[held] - dist[held]).mean(), rel=1e-9)
            res[key][0].append(hold_mae)
            res[key][1].append(np.abs(ed - dist).mean())
    for k in (0, 1):
        gpu, cpu = np.array(res["gpu"][k]), np.array(res["cpu"][k])
        se = np.sqrt(gpu.var(ddof=1) / 10 + cpu.var(ddof=1) / 10)
        assert abs(gpu.mean() - cpu.mean()) <= max(2 * se, 0.03 * cpu.mean()), (k, gpu, cpu)


# ------------------------------------------------------------------ edge cases ---------------
def test_degenerate_inputs_stay_finite():
    # tests/testthat/test-edge-cases.R:5-82,243-263
    zero = np.zeros((3, 3))
    with pytest.warns(UserWarning, match="No finite non-zero dissimilarities"):
        r = core.euclidean_embedding(zero, 2, 20, 1.0, 0.01, 0.01)
    assert np.isfinite(r.mae)
    thr = np.array([["0", ">5", "<10"], [">5", "0", ">20"], ["<10", ">20", "0"]], dtype=object)
    r = core.euclidean_embedding(thr, 2, 30, 2.0, 0.01, 0.05)
    assert np.all(np.isfinite(r.positions)) and np.all(np.isfinite(r.est_distances))
    one = np.full((4, 4), np.nan); one[0, 1] = one[1, 0] = 5; np.fill_diagonal(one, 0)
    r = core.euclidean_embedding(one, 2, 50, 1.0, 0.01, 0.1)
    assert np.all(np.isfinite(r.positions))
    rng = np.random.default_rng(0)
    for lo, hi in ((1000, 10000), (1e-6, 1e-3)):
        m = rng.uniform(lo, hi, size=(3, 3)); m = np.triu(m, 1); m = m + m.T
        r = core.euclidean_embedding(m, 2, 20, 1.0, 0.01, 0.01)
        assert np.all(np.isfinite(r.positions))
    m = rng.uniform(1, 10, size=(5, 5)); m = np.triu(m, 1); m = m + m.T
    r = core.euclidean_embedding(m, 4, 30, 0.1, 0.001, 0.001)
    assert np.all(np.isfinite(r.positions))


def test_numerical_instability_is_reported_like_rcpp_stop():
    # src/optimization.cpp:359-361
    init = np.zeros((4, 2))
    for mode, prec, big in ((_lib.MODE_REPLAY, 0, True), (_lib.MODE_COLOURED, _lib.PREC_F64_EXACT, True),
                            (_lib.MODE_COLOURED, _lib.PREC_F32, False)):
        with pytest.raises(_lib.TopolowError) as e:
            _lib.fit(init, [2, 2, 1, 1], [0], [1], [1.0], [0], 20, 1e300 if big else 1e30, 0.01, 1e308 if big else 1e38,
                     convergence_window=100, convergence_check_freq=50, mode=mode, precision=prec)
        assert e.value.status == _lib.ERR_NONFINITE
        assert "Numerical instability at iteration 10. Reduce k0 or c_repulsion." in str(e.value)


def test_bad_arguments_are_rejected():
    args = list(small_problem(20, 2, 0.5, 0))
    bad = list(args); bad[2] = np.array(args[2]); bad[2][0] = 99
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(*bad, 5, 1.0, 0.01, 0.01)
    assert e.value.status == _lib.ERR_BAD_ARG and "edge index" in str(e.value)
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(np.zeros((20, 17)), *args[1:], 5, 1.0, 0.01, 0.01)
    assert e.value.status == _lib.ERR_BAD_ARG


def test_sixteen_argument_entry_point():
    # the flattened .Call signature (src/RcppExports.cpp:16-39)
    init, deg, ei, ej, ed, et = small_problem(40, 2, 0.4, 3)
    n = 40
    dm, tm = cpu_oracle.dense_from_edges(n, ei, ej, ed, et)
    out = np.empty((n, 2), order="F")
    conv, iters = C.c_int32(0), C.c_int32(0)
    mae, k = C.c_double(0), C.c_double(0)
    msg = C.create_string_buffer(256)
    initf = np.asfortranarray(init)
    dmf, tmf = np.asfortranarray(dm), np.asfortranarray(tm.astype(np.int32))
    rc = _lib.lib().topolow_optimize_layout_exact(
        initf.ctypes.data_as(_lib._dp), n, 2, dmf.ctypes.data_as(_lib._dp), tmf.ctypes.data_as(_lib._i32p),
        deg.ctypes.data_as(_lib._i32p), ei.ctypes.data_as(_lib._i32p), ej.ctypes.data_as(_lib._i32p),
        ed.ctypes.data_as(_lib._dp), et.ctypes.data_as(_lib._i32p), len(ei), 30, 2.0, 0.01, 0.01, 1e-4, 5, 3, 0,
        out.ctypes.data_as(_lib._dp), C.byref(conv), C.byref(iters), C.byref(mae), C.byref(k), msg, 256)
    assert rc == 0 and np.all(np.isfinite(out)) and 0 < iters.value <= 30 and mae.value > 0


# ------------------------------------------------------------------ R-facing mirror -----------
def test_euclidean_embedding_object_and_post_processing():
    # tests/testthat/test-core.R:67-139
    m = random_r_matrix(30, 0.5, 11)
    names = ["P%d" % i for i in range(30)]
    init = np.random.default_rng(2).normal(size=(30, 2))
    r = core.euclidean_embedding(m, 2, 40, 1.0, 0.01, 0.01, initial_positions=init, rownames=names, precision="f64")
    assert set(r) >= {"positions", "est_distances", "mae", "iter", "parameters", "convergence"}
    assert r.positions.shape == (30, 2) and isinstance(r.convergence["achieved"], bool)
    assert r.parameters["method"] == core.METHOD_NAME and sorted(r.rownames) == sorted(names)
    np.testing.assert_allclose(r.est_distances, r_glue.dist_matrix(r.positions), rtol=0, atol=0)
    # mae of R/core.R:479-481 against the oracle's restatement on the same (reordered) matrix
    mm = m if r.order is None else m[np.ix_(r.order, r.order)]
    raw = np.array([[r_glue._as_numeric(x) for x in row] for row in mm])
    ok = ~np.isnan(raw)
    assert r.mae == pytest.approx(float(np.mean(np.abs(raw[ok] - r.est_distances[ok]))), rel=1e-12)
    # thresholds + NA (test-core.R:90-104)
    t = np.array([[0, ">2", None], [">2", 0, 4], [None, 4, 0]], dtype=object)
    r = core.euclidean_embedding(t, 2, 10, 1.0, 0.01, 0.01)
    assert np.isfinite(r.est_distances[0, 2]) and r.est_distances[0, 2] == r.est_distances[2, 0]
    # triangle relations (test-core.R:106-127)
    tri = np.array([[0, 1, 2], [1, 0, 1], [2, 1, 0]], dtype=float)
    r = core.euclidean_embedding(tri, 2, 10, 1.0, 0.01, 0.01, preserve_order=True)
    dd = r.est_distances
    assert dd[0, 2] > dd[0, 1] and dd[0, 2] < dd[0, 1] + dd[1, 2]


def test_holdout_errors_and_likelihood_function():
    rng = np.random.default_rng(3)
    pos = rng.normal(size=(25, 3))
    ci = rng.integers(0, 25, size=200).astype(np.int32); cj = rng.integers(0, 25, size=200).astype(np.int32)
    truth = rng.uniform(0, 5, size=200); truth[::17] = np.nan
    s, c = _lib.holdout_errors(pos, ci, cj, truth)
    d = np.linalg.norm(pos[ci] - pos[cj], axis=1)
    ok = ~np.isnan(truth)
    assert c == ok.sum() and s == pytest.approx(np.abs(truth[ok] - d[ok]).sum(), rel=1e-12)
    # likelihood_function: same folds and initial positions, FP64 -> pooled numbers of the same size
    m = random_r_matrix(26, 0.7, 5)
    folds = r_glue.make_folds(m, 4, np.random.default_rng(1))
    inits = [[np.random.default_rng(10 + f).normal(size=(26, 2)) for f in range(4)]]
    want = r_glue.likelihood_function(m, 60, 1e-4, 2, 2.0, 0.02, 0.01, folds=4, fold_indices=folds, init_list=inits[0])
    got = cv.likelihood_function(m, 60, 1e-4, 2, 2.0, 0.02, 0.01, folds=4, fold_indices=folds, init_list=inits,
                                 precision="f64")
    assert [f["n_samples"] for f in got["folds"]] == [f["n_samples"] for f in want["folds"]]
    assert got["Holdout_MAE"] == pytest.approx(want["Holdout_MAE"], rel=0.25)   # different pair orders
    assert got["NLL"] == pytest.approx(sum(f["n_samples"] for f in got["folds"]) * (1 + np.log(2 * got["Holdout_MAE"])))
    # the same comparison with the pair order taken out of it: the CPU side replays, fold by fold, the sequential
    # order the GPU schedule is equivalent to (FP64 both sides) - every pooled number then agrees to rounding
    value, code, is_na = core.parse_dissimilarity(m)
    orders = []
    for f, hold in enumerate(folds):
        prob = cv._fold_job(value, code, is_na, np.asarray(hold), True)[0]
        plan = _lib.Plan(inits[0][f], prob["degrees"], prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"],
                         60, 2.0, 0.02, 0.01, 1e-4, 5, 3, precision=_lib.PREC_F64_EXACT, seed=f)
        orders.append(np.stack([plan.enumerate(it) for it in range(60)]))
        plan.close()
    want2 = r_glue.likelihood_function(m, 60, 1e-4, 2, 2.0, 0.02, 0.01, folds=4, fold_indices=folds, init_list=inits[0],
                                       pair_orders=orders)
    assert got["Holdout_MAE"] == pytest.approx(want2["Holdout_MAE"], rel=1e-9)
    assert got["NLL"] == pytest.approx(want2["NLL"], rel=1e-9)
    assert [f["iter"] for f in got["folds"]] == [f["iter"] for f in want2["folds"]]
    assert [f["sum_abs_errors"] for f in got["folds"]] == pytest.approx([f["sum_abs_errors"] for f in want2["folds"]], rel=1e-9)


def test_batch_equals_individual_fits():
    jobs, singles = [], []
    for j, (n, d) in enumerate([(40, 2), (150, 3), (90, 5), (285, 5)]):
        a = small_problem(n, d, 0.2, 50 + j)
        kw = dict(n_iter=25, k0=3.0, cooling_rate=0.02, c_repulsion=0.01, seed=j)
        jobs.append(dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4],
                         edge_thresh=a[5], **kw))
        singles.append(_lib.fit(*a, 25, 3.0, 0.02, 0.01, seed=j))
    jobs.append(dict(initial_positions=np.zeros((1, 2)), degrees=[1], edge_i=[], edge_j=[], edge_dist=[],
                     edge_thresh=[], n_iter=5, k0=1.0, cooling_rate=0.1, c_repulsion=0.1))
    out = _lib.fit_batch(jobs)
    for got, want in zip(out[:4], singles):
        assert np.array_equal(got["positions"], want["positions"]) and got["iterations"] == want["iterations"]
    assert out[4]["status"] == _lib.ERR_TOO_FEW_POINTS      # per-job status, the batch itself succeeds


def test_cv_grid_batch_shares_fold_records_and_launches():
    # >= 16 jobs: one CTA per fit, many fits per launch (grouped by ndim / precision), and the jobs that
    # point at the same edge arrays share one set of device records.  None of that may change a result:
    # every job equals the same fit run alone with the same geometry (one CTA, 64-point tiles).
    a = small_problem(300, 4, 0.3, 91)
    b = small_problem(300, 4, 0.3, 92)
    rng = np.random.default_rng(5)
    jobs, want = [], []
    for j in range(18):
        src = a if j % 2 == 0 else b            # two "folds", shared by reference across the samples
        d = 2 + j % 3
        prec = _lib.PREC_F64_EXACT if j % 6 == 5 else _lib.PREC_F32
        init = rng.normal(size=(300, d))
        kw = dict(n_iter=12, k0=2.0 + j, cooling_rate=0.02, c_repulsion=0.01, seed=100 + j, precision=prec)
        jobs.append(dict(initial_positions=init, degrees=src[1], edge_i=src[2], edge_j=src[3], edge_dist=src[4],
                         edge_thresh=src[5], **kw))
        want.append(_lib.fit(init, src[1], src[2], src[3], src[4], src[5], 12, 2.0 + j, 0.02, 0.01, seed=100 + j,
                             precision=prec, max_ctas=1, tile_points=64))
    out = _lib.fit_batch(jobs)
    for got, ref in zip(out, want):
        assert got["status"] == _lib.OK
        assert np.array_equal(got["positions"], ref["positions"])
        assert got["final_mae"] == ref["final_mae"] and got["iterations"] == ref["iterations"]
    # the same batch with private copies of the edge arrays (nothing shared) gives the same bits
    copies = [dict(j, edge_i=np.array(j["edge_i"]), edge_j=np.array(j["edge_j"]), edge_dist=np.array(j["edge_dist"]),
                   edge_thresh=np.array(j["edge_thresh"])) for j in jobs]
    for got, ref in zip(_lib.fit_batch(copies), out):
        assert np.array_equal(got["positions"], ref["positions"])


def test_holdout_scored_inside_the_fit_equals_the_separate_kernel():
    # topolow_problem.holdout_*: same numbers as topolow_holdout_errors on the returned positions
    a = small_problem(220, 3, 0.25, 17)
    rng = np.random.default_rng(3)
    ci, cj = rng.integers(0, 220, 500).astype(np.int32), rng.integers(0, 220, 500).astype(np.int32)
    truth = rng.uniform(0.5, 9.0, 500)
    truth[::37] = np.nan                                   # NA truth cells are dropped
    for kw in (dict(), dict(precision=_lib.PREC_F64_EXACT), dict(mode=_lib.MODE_REPLAY)):
        r = _lib.fit(*a, 15, 3.0, 0.02, 0.01, seed=4, holdout=(ci, cj, truth), **kw)
        s_abs, cnt = _lib.holdout_errors(r["positions"], ci, cj, truth)
        assert r["holdout_count"] == cnt == int(np.sum(~np.isnan(truth)))
        assert r["holdout_sum_abs"] == s_abs
        d = np.linalg.norm(r["positions"][ci] - r["positions"][cj], axis=1)
        assert s_abs == pytest.approx(np.nansum(np.abs(truth - d)), rel=1e-12)
    jobs = [dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4], edge_thresh=a[5],
                 n_iter=15, k0=3.0, cooling_rate=0.02, c_repulsion=0.01, seed=s, holdout=(ci, cj, truth)) for s in range(17)]
    for r in _lib.fit_batch(jobs):
        s_abs, cnt = _lib.holdout_errors(r["positions"], ci, cj, truth)
        assert (r["holdout_sum_abs"], r["holdout_count"]) == (s_abs, cnt)
    with pytest.raises(_lib.TopolowError):
        _lib.fit(*a, 2, 3.0, 0.02, 0.01, holdout=(np.array([220], dtype=np.int32), np.array([0], dtype=np.int32), np.array([1.0])))


# ------------------------------------------------------------------ full-size properties ------
def test_cfg3_size_fp32_against_fp64_and_pair_count():
    prob = synth.make_problem(10_000, 10, 0.95, seed=1)
    fa = synth.fit_args(prob)
    hp = (5.0, 0.01, 0.02, 1e-4, 100, 3)
    a = _lib.fit(*fa, 3, *hp, precision=_lib.PREC_F64_EXACT, seed=2, tile_points=64)
    b = _lib.fit(*fa, 3, *hp, precision=_lib.PREC_F32, seed=2, tile_points=64, max_warps=4)   # the FP64 schedule
    assert a["pair_updates"] == b["pair_updates"] == 3 * 10_000 * 9_999 // 2
    assert np.abs(a["positions"] - b["positions"]).max() <= 1e-3 * np.abs(a["positions"]).max()
    assert b["final_mae"] == pytest.approx(a["final_mae"], rel=1e-3)


def test_cfg4_size_runs_and_improves():
    prob = synth.make_problem(100_000, 16, 0.99, seed=0)
    fa = synth.fit_args(prob)
    r = _lib.fit(*fa, 6, 5.0, 0.01, 0.02, 1e-4, 100, 3, seed=0, trace=True)
    assert r["pair_updates"] == 6 * 100_000 * 99_999 // 2 and np.all(np.isfinite(r["positions"]))
    t = r["trace_mae"][~np.isnan(r["trace_mae"])]
    assert len(t) == 2 and t[1] < t[0]


# ------------------------------------------------------------------ through the .Call shim -------
SHIM_SEED = (2 ** 30 << 32) | 2 ** 31      # what integration/r_shim.c draws from the stand-in unif_rand stream (0.25, 0.5)


def _shim(exe, *args):
    import json
    import subprocess
    out = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_r_shim_against_the_real_library(tmp_path):
    """integration/r_shim.c compiled against the stand-in R headers and linked with libtopolow_b200.so: what R's
    .Call would get back equals the C ABI driven through ctypes with the same inputs and seed, bit for bit (single
    fit in the coloured and the row-block mode, a batch with hold-out cells), an interrupt comes back as
    TOPOLOW_ERR_INTERRUPTED and is raised from the shim, a non-finite fit carries the reference's message."""
    from conftest import build_r_shim_harness, write_problem_bin
    exe = build_r_shim_harness(str(tmp_path / "harness_gpu"), real_library=True)
    init, deg, ei, ej, ed, et = small_problem(300, 3, 0.1, 21)
    held = np.random.default_rng(1).random(len(ei)) < 0.1
    hold = (ei[held], ej[held], ed[held])
    train = (init, deg, ei[~held], ej[~held], ed[~held], et[~held])
    write_problem_bin(tmp_path / "p.bin", *train, hold)
    for mode_name, mode in (("coloured", _lib.MODE_COLOURED), ("rowblock", _lib.MODE_ROWBLOCK)):
        r = _shim(exe, "single", tmp_path / "p.bin", tmp_path / "o.bin", 60, 5.0, 0.01, 0.02, 1e-4, 5, 3, mode_name)
        assert r["protect_depth"] == 0 and r["type_errors"] == 0 and r["rng_violations"] == 0
        out = np.fromfile(tmp_path / "o.bin")
        want = _lib.fit(*train, 60, 5.0, 0.01, 0.02, 1e-4, 5, 3, mode=mode, seed=SHIM_SEED)
        assert (bool(out[0]), int(out[1]), out[2], out[3]) == (want["converged"], want["iterations"], want["final_mae"], want["final_k"])
        assert np.array_equal(out[4:].reshape(3, 300).T, want["positions"])
    r = _shim(exe, "batch", tmp_path / "p.bin", tmp_path / "b.bin", 3, 40, 4.0, 0.01, 0.02, 1e-4, 5, 3, 1)
    assert [j["status"] for j in r["jobs"]] == [0, 0, 0] and r["protect_depth"] == 0
    got = np.fromfile(tmp_path / "b.bin").reshape(3, 7 + 900)
    jobs = [dict(initial_positions=train[0], degrees=train[1], edge_i=train[2], edge_j=train[3], edge_dist=train[4],
                 edge_thresh=train[5], n_iter=40, k0=4.0 * (1 + 0.25 * j), cooling_rate=0.01, c_repulsion=0.02,
                 relative_epsilon=1e-4, convergence_window=5, convergence_check_freq=3, seed=SHIM_SEED + j, holdout=hold)
            for j in range(3)]
    want = _lib.fit_batch(jobs)
    for j in range(3):
        assert got[j, 2] == want[j]["final_mae"] and got[j, 4] == want[j]["holdout_sum_abs"] and got[j, 5] == want[j]["holdout_count"]
        assert np.array_equal(got[j, 7:].reshape(3, 300).T, want[j]["positions"])
    r = _shim(exe, "interrupt", tmp_path / "p.bin", 2)          # second poll = after the first 50-iteration chunk
    assert r["left_by"] == "Rf_onintr" and r["raw_interrupt_jumps"] == 0 and r["interrupt_checks"] == 2
    r = _shim(exe, "too_few")
    assert r["left_by"] == "Rf_error" and r["message"] == "Need at least 2 points for embedding"


def test_interruptible_fit_releases_everything():
    """topolow_fit_interruptible: a callback that fires at chunk k ends the fit with status 5; device memory in use
    returns to its level (no leaked plan, stream or buffer over 20 interrupted fits)."""
    import torch
    args = small_problem(600, 4, 0.05, 8)
    free0 = None
    for rep in range(21):
        calls = []
        with pytest.raises(_lib.TopolowError) as e:
            _lib.fit(*args, 400, 5.0, 0.01, 0.02, 1e-12, 1000, 3, interrupt=lambda: (calls.append(1), len(calls) > 2)[1])
        assert e.value.status == _lib.ERR_INTERRUPTED and len(calls) == 3
        torch.cuda.synchronize()
        if rep == 0:
            free0 = torch.cuda.mem_get_info()[0]
    assert torch.cuda.mem_get_info()[0] >= free0 - (8 << 20)


# ------------------------------------------------------------------ BASELINE.json configs[0..2] ---
PUBLISHED = {   # inst/examples/methods-comparison-h3n2-hiv-denv.Rmd:312-331 (k0, cooling_rate, c_repulsion), ndim 5
    "h3n2": (14.76214, 0.03641074, 0.002943064),
    "hiv": (3.550036, 0.04130713, 0.0007038619),
}


def _parity(gpu, cpu, rel):
    gpu, cpu = np.asarray(gpu), np.asarray(cpu)
    se = np.sqrt(gpu.var(ddof=1) / len(gpu) + cpu.var(ddof=1) / len(cpu))
    assert abs(gpu.mean() - cpu.mean()) <= max(2 * se, rel * cpu.mean()), (gpu.mean(), cpu.mean(), se, gpu, cpu)


@pytest.mark.parametrize("name", ["h3n2", "hiv"])
def test_coloured_parity_on_the_bundled_maps(name):
    """configs[0] / configs[1]: the bundled H3N2 and HIV tables (HIV with '>' thresholds), ndim 5, mapping_max_iter
    1000, published hyper-parameters, 10 % of the exact cells held out, 10 seeds: the production schedule in FP32
    vs the reference's std::shuffle loop - edge MAE at the best state and held-out MAE within max(2 SE, 3 %)."""
    p = load_fixture(name)
    n = int(p["n"])
    ei, ej, ed, et = p["edge_i"], p["edge_j"], p["edge_dist"], p["edge_thresh"]
    k0, cool, crep = PUBLISHED[name]
    mae, hold = ([], []), ([], [])
    for seed in range(10):
        rng = np.random.default_rng(100 + seed)
        held = (rng.random(len(ei)) < 0.1) & (et == 0)
        tr = ~held
        deg_tr = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
        init = np.vstack([np.zeros((1, 5)), np.cumsum(rng.uniform(0, 2 * ed[et == 0].max() / n, size=(n - 1, 5)), axis=0)])
        train = (init, deg_tr, ei[tr], ej[tr], ed[tr], et[tr], 1000, k0, cool, crep, 1e-4, 5, 3)
        g = _lib.fit(*train, seed=seed)
        c = cpu_oracle.optimize_layout_exact(*train, seed=seed)
        for k, r in enumerate((g, c)):
            dist = np.linalg.norm(r["positions"][ei] - r["positions"][ej], axis=1)
            mae[k].append(r["final_mae"])
            hold[k].append(np.abs(ed[held] - dist[held]).mean())
    _parity(mae[0], mae[1], 0.03)
    _parity(hold[0], hold[1], 0.03)


def _cfg3_problem():
    """The problem tools/make_golden_cfg3.py ran the reference loop on (same generator, seeds and hold-out)."""
    import json
    import os
    from conftest import GOLDEN
    gold = json.load(open(os.path.join(GOLDEN, "cfg3_reference_loop.json")))
    n, d = gold["n"], gold["ndim"]
    prob = synth.make_problem(n, d, gold["missing"], seed=gold["synth_seed"])
    ei, ej, ed, et = prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"]
    held = (np.random.default_rng(gold["holdout_seed"]).random(len(ei)) < 0.10) & (et == 0)
    tr = ~held
    assert int(tr.sum()) == gold["train_edges"] and int(held.sum()) == gold["heldout_cells"]
    deg = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
    hp = gold["hyper"]
    train = (prob["initial_positions"], deg, ei[tr], ej[tr], ed[tr], et[tr], gold["iterations"], hp["k0"], hp["cooling_rate"],
             hp["c_repulsion"], hp["relative_epsilon"], hp["convergence_counter"], hp["convergence_check_freq"])
    return gold, train, (ei[held], ej[held], ed[held])


@pytest.mark.parametrize("mode", ["coloured", "rowblock"])
def test_cfg3_against_the_reference_loop_goldens(mode):
    """configs[2] at full size (10 000 points, 95 % missing, ndim 10, thresholds, 100 iterations, 10 % of the exact
    cells held out): three seeds of the GPU schedule against three seeds of the reference's dense std::shuffle loop
    (tests/golden/cfg3_reference_loop.json, 23 CPU-minutes per seed, made by tools/make_golden_cfg3.py): edge MAE at the
    best state, held-out MAE and the MAE trace every 15 iterations within 2 %.  For the coloured mode this is also the check that a point -> tile
    placement fixed for the whole fit (plan.cu kLayoutSeed; tile -> super-block placement, round order and ring strides
    are re-drawn every iteration) is statistically the same process as a fresh shuffle of all pairs at this size."""
    gold, train, (hi, hj, ht) = _cfg3_problem()
    ref_mae = np.array([r["final_mae"] for r in gold["runs"]])
    ref_hold = np.array([r["heldout_mae"] for r in gold["runs"]])
    ref_trace = np.mean([r["mae_trace"] for r in gold["runs"]], axis=0)
    maes, holds = [], []
    for seed in range(3):
        g = _lib.fit(*train, mode=_lib.MODE_ROWBLOCK if mode == "rowblock" else _lib.MODE_COLOURED, seed=seed, trace=True)
        assert g["iterations_run"] == gold["iterations"]
        dist = np.linalg.norm(g["positions"][hi] - g["positions"][hj], axis=1)
        maes.append(g["final_mae"]); holds.append(np.abs(ht - dist).mean())
        tr = g["trace_mae"][~np.isnan(g["trace_mae"])]
        assert len(tr) == len(ref_trace)
        # iterations 15, 30, ..., 90 (the first checks are the steep part).  The row-block scheme is Jacobi across points and
        # lags the sequential loop while the map unfolds (measured at iteration 15: 2.79 vs 2.51), from iteration 30 on
        # it is the same curve
        if mode == "rowblock":
            np.testing.assert_allclose(tr[4], ref_trace[4], rtol=0.15)
            np.testing.assert_allclose(tr[9::5], ref_trace[9::5], rtol=0.02)
        else:
            np.testing.assert_allclose(tr[4::5], ref_trace[4::5], rtol=0.02)
    assert np.mean(maes) == pytest.approx(ref_mae.mean(), rel=0.02), (maes, ref_mae)
    assert np.mean(holds) == pytest.approx(ref_hold.mean(), rel=0.02), (holds, ref_hold)


@pytest.mark.skipif("__import__('torch').cuda.device_count() < 2")
def test_exact_sharded_map_over_nccl_equals_the_emulation(tmp_path):
    """Two processes, two GPUs, NCCL: the exact row-sharded map (topolow_b200/sharded.py) equals its single-GPU
    emulation bit for bit (tools/gpu_sharded_check.py asserts it on every rank)."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "gpu_sharded_check.py"), "3000", "6", "0.95", "2"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]


def test_sparse_table_entry_equals_the_matrix_entry():
    """euclidean_embedding_coo (nothing n x n is built) returns the positions, convergence fields and mae of
    euclidean_embedding on the matrix the table stands for; est_distances on the listed pairs and on extra
    (held-out) pairs equal the dense est_distances there."""
    m = random_r_matrix(90, 0.3, 5)
    ii, jj = np.nonzero(np.frompyfunc(lambda x: x is not None, 1, 1)(m).astype(bool))
    up = ii < jj
    init = np.random.default_rng(2).normal(size=(90, 3))
    for preserve in (True, False):
        dense = core.euclidean_embedding(m, 3, 80, 4.0, 0.02, 0.01, initial_positions=init, preserve_order=preserve, seed=3)
        sp = core.euclidean_embedding_coo(90, ii[up], jj[up], m[ii[up], jj[up]], 3, 80, 4.0, 0.02, 0.01, initial_positions=init,
                                          preserve_order=preserve, seed=3, extra_pairs=(np.array([0, 5, 7]), np.array([9, 1, 8])))
        assert np.array_equal(dense["positions"], sp["positions"])
        assert dense["convergence"] == sp["convergence"] and dense["iter"] == sp["iter"]
        assert sp["mae"] == pytest.approx(dense["mae"], rel=1e-9)
        ci, cj = sp["pairs"]
        np.testing.assert_allclose(sp["est_distances"], dense["est_distances"][ci, cj], rtol=1e-12)
        order = dense["order"] if dense["order"] is not None else np.arange(90)
        rank = np.empty(90, dtype=int); rank[order] = np.arange(90)
        np.testing.assert_allclose(sp["est_extra"], dense["est_distances"][rank[[0, 5, 7]], rank[[9, 1, 8]]], rtol=1e-12)


# ------------------------------------------------------------------ measurement graph, sparse CV --
def test_device_components_equal_scipy():
    """topolow_components (csrc/graph.cu) vs scipy's connected_components: component count, selected points and
    selected edges for random graphs, every point / many candidate masks, isolated points, no edges at all."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    rng = np.random.default_rng(0)
    for n, dens, n_masks in ((50, 0.03, 7), (400, 0.004, 16), (3000, 0.0006, 5), (2000, 0.01, 3), (10, 0.0, 2)):
        iu = np.triu_indices(n, 1)
        keep = rng.random(len(iu[0])) < dens
        ei, ej = iu[0][keep].astype(np.int32), iu[1][keep].astype(np.int32)
        if len(ei) and rng.random() < 0.5:
            ei, ej = np.r_[ei, ej[:5]], np.r_[ej, ei[:5]]           # duplicates and reversed orientation are legal
        masks = rng.random((n_masks, n)) < 0.6
        masks[0, :] = True
        for mk_set in (None, masks):
            comp, pts, edg = _lib.components(n, ei, ej, mk_set)
            for a, mk in enumerate(np.ones((1, n), bool) if mk_set is None else mk_set):
                k = mk[ei] & mk[ej]
                lab = connected_components(coo_matrix((np.ones(k.sum()), (ei[k], ej[k])), shape=(n, n)), directed=False)[1]
                assert comp[a] == len(set(lab[mk])) and pts[a] == mk.sum() and edg[a] == k.sum(), (n, a)
    with pytest.raises(_lib.TopolowError):
        _lib.components(5, [0, 9], [1, 2])


def test_subsampling_on_the_device_follows_the_reference_loop():
    from topolow_b200 import subsample
    m = random_r_matrix(200, 0.03, 4, thresholds=False)
    fm = np.array([[np.nan if x is None else float(x) for x in row] for row in m])
    np.fill_diagonal(fm, 0.0)
    import warnings as w
    with w.catch_warnings():
        w.simplefilter("ignore")
        full = subsample.check_matrix_connectivity(fm)
        assert full["n_components"] == r_glue.check_matrix_connectivity(fm)["n_components"]
        found = 0
        for seed in range(8):
            rng = np.random.default_rng(seed)
            attempts = [np.sort(rng.choice(200, size=120, replace=False)) for _ in range(5)]
            want = r_glue.subsample_dissimilarity_matrix(fm, attempts)
            try:
                got = subsample.subsample_dissimilarity_matrix(fm, 120, rng=np.random.default_rng(seed), preserve_order=True)
            except RuntimeError:
                assert want is None
                continue
            found += 1
            assert got["attempt_number"] == want[0] and np.array_equal(got["selected_indices"], want[1])
            assert got["completeness"] == pytest.approx(want[2]["completeness"])
    assert found > 0


def test_likelihood_on_a_table_equals_likelihood_on_the_matrix():
    """likelihood_batch_coo (folds drawn and masked on the cell list, nothing n x n) == likelihood_batch on the matrix
    for the same drawn cells and initial positions: every pooled number and every fold row."""
    n = 80
    m = random_r_matrix(n, 0.3, 9)
    value, code, is_na = core.parse_dissimilarity(m)
    ii, jj = np.nonzero(np.triu(~is_na, 1))
    full = core.build_problem_coo(n, ii, jj, m[ii, jj], preserve_order=True)
    cells = cv.make_folds_cells(n, full["cell_i"], full["cell_j"], 4, np.random.default_rng(1))
    lin = []
    for picks in cells:
        a = np.where(picks < n, picks, full["cell_i"][np.maximum(picks - n, 0) >> 1])
        b = np.where(picks < n, picks, full["cell_j"][np.maximum(picks - n, 0) >> 1])
        swap = (picks >= n) & (((picks - n) & 1) == 1)
        a, b = np.where(swap, b, a), np.where(swap, a, b)
        lin.append(a + b * n)
    samples = [dict(N=2, k0=3.0, cooling_rate=0.02, c_repulsion=0.01), dict(N=4, k0=6.0, cooling_rate=0.01, c_repulsion=0.02)]
    rng = np.random.default_rng(5)
    inits = [[rng.normal(size=(n, s["N"])) for _ in range(4)] for s in samples]
    dense = cv.likelihood_batch(m, samples, 60, 1e-4, folds=4, fold_indices=lin, init_list=inits, seed=2)
    table = cv.likelihood_batch_coo(n, ii, jj, m[ii, jj], samples, 60, 1e-4, folds=4, fold_cells=cells, init_list=inits, seed=2)
    for d, t in zip(dense, table):
        assert d["Holdout_MAE"] == pytest.approx(t["Holdout_MAE"], rel=1e-12) and d["NLL"] == pytest.approx(t["NLL"], rel=1e-12)
        assert [f["n_samples"] for f in d["folds"]] == [f["n_samples"] for f in t["folds"]]
        assert [f["iter"] for f in d["folds"]] == [f["iter"] for f in t["folds"]]


def test_batched_adaptive_chains_on_the_device():
    """sampler.adaptive_mc_batch: 4 chains x 2 rounds, every round one likelihood_batch call of chains x folds fits on
    the device; the table grows by valid rows whose MAE is that of the drawn parameters."""
    from topolow_b200 import sampler
    m = random_r_matrix(60, 0.4, 3, thresholds=False)
    rng = np.random.default_rng(0)
    design = sampler.lhs_design(12, (2, 4), (1.0, 8.0), (1e-3, 0.05), (0.005, 0.05), rng=rng)
    sets = [dict(N=int(design["N"][i]), k0=design["k0"][i], cooling_rate=design["cooling_rate"][i], c_repulsion=design["c_repulsion"][i])
            for i in range(12)]
    first = cv.likelihood_batch(m, sets, 80, 1e-4, folds=4, rng=rng)
    table = {"log_N": np.log(design["N"]), "log_k0": np.log(design["k0"]), "log_cooling_rate": np.log(design["cooling_rate"]),
             "log_c_repulsion": np.log(design["c_repulsion"]), "Holdout_MAE": np.array([r["Holdout_MAE"] for r in first]),
             "NLL": np.array([r["NLL"] for r in first]), "mean_iter": np.array([r["mean_iter"] for r in first]),
             "pct_converged": np.array([r["pct_converged"] for r in first])}
    assert np.all(np.isfinite(table["Holdout_MAE"]))
    grown = sampler.adaptive_mc_batch(table, m, iterations=2, chains=4, mapping_max_iter=80, relative_epsilon=1e-4, folds=4, rng=rng)
    assert len(grown["Holdout_MAE"]) == 12 + 8 and np.all(np.isfinite(grown["Holdout_MAE"])) and np.all(grown["Holdout_MAE"] > 0)
    np.testing.assert_allclose(grown["NLL"][12:] / (1 + np.log(2 * grown["Holdout_MAE"][12:])),
                               np.round(grown["NLL"][12:] / (1 + np.log(2 * grown["Holdout_MAE"][12:]))), atol=1e-6)   # NLL = n (1 + log 2 MAE)


def test_repeated_runs_are_bit_identical():
    """Race canary (compute-sanitizer is closed on the GPU pool): the protocols that could race - tile hand-off between
    warps through shared-memory flags, release / acquire round counters between CTAs, the grid barrier, the many-fits
    kernel, row-block epoch flags and peer stores between three shards - give the same bits 20 times in a row."""
    from topolow_b200 import rowblock
    args = small_problem(1500, 3, 0.03, 12)
    hp = (5.0, 0.02, 0.02, 1e-4, 5, 2)
    first = None
    for _ in range(20):
        r = _lib.fit(*args, 12, *hp, seed=5, tile_points=32)
        first = first if first is not None else r
        assert np.array_equal(r["positions"], first["positions"]) and r["final_mae"] == first["final_mae"]
    a = small_problem(200, 4, 0.1, 2)
    jobs = [dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4], edge_thresh=a[5], n_iter=20,
                 k0=3.0 + j, cooling_rate=0.02, c_repulsion=0.01, seed=j) for j in range(20)]
    ref = _lib.fit_batch(jobs)
    for _ in range(5):
        again = _lib.fit_batch(jobs)
        assert all(np.array_equal(x["positions"], y["positions"]) for x, y in zip(ref, again))
    b = small_problem(1300, 5, 0.04, 6)
    first = None
    for _ in range(20):
        ls = rowblock.LocalShards(*b, 9, *hp, n_ranks=3, seed=2)
        ls.run(9)
        r = ls.result(rank=2)
        ls.close()
        first = first if first is not None else r
        assert np.array_equal(r["positions"], first["positions"]) and r["final_mae"] == first["final_mae"]
