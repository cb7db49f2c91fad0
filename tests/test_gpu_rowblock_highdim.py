"""GPU tests of the row-block mode at ndim 17..32 (topolow_b200/csrc/rowblock.cu, H = 10, 12, 14, 16: the row padded to a
multiple of four coordinates, the pad computed on as zeros; the FP32 difference form of the repulsion pass only).
Everything goes through the C ABI, as in test_gpu_rowblock.py, with the same bars."""
import numpy as np
import pytest

from conftest import small_problem
from oracle import cpu_oracle
from topolow_b200 import _lib, core, rowblock

pytestmark = pytest.mark.gpu

HP = (5.0, 0.01, 0.02, 1e-4, 5, 3)


# ------------------------------------------------------------------ numerics ---------------------
@pytest.mark.parametrize("n,d,dens", [(600, 17, 0.08), (900, 20, 0.05), (700, 24, 0.06), (1100, 27, 0.04), (2100, 32, 0.02)])
def test_rowblock_highdim_tracks_its_fp64_restatement(n, d, dens):
    args = small_problem(n, d, dens, 10 * n + d, thresholds=True)
    sop = rowblock.slot_order(n)
    want = cpu_oracle.relaxed_optimize_layout(*args, 6, *HP, seed=4, slot_of_point=sop)
    got = _lib.fit(*args, 6, *HP, mode=_lib.MODE_ROWBLOCK, seed=4)
    assert got["positions"].shape == (n, d)
    scale = max(np.abs(want["positions"]).max(), 1.0)
    err = np.abs(got["positions"] - want["positions"])
    assert np.quantile(err, 0.99) <= 2e-4 * scale and err.max() <= 2e-3 * scale, (np.quantile(err, 0.99), err.max(), scale)
    assert got["final_mae"] == pytest.approx(want["final_mae"], rel=1e-3)
    assert got["iterations"] == want["iterations"] and got["iterations_run"] == 6
    assert got["final_k"] == pytest.approx(want["final_k"], rel=1e-12)
    assert got["pair_updates"] == 6 * n * (n - 1) // 2


def test_rowblock_highdim_controller_and_trace_follow_the_restatement():
    args = small_problem(500, 24, 0.2, 77, thresholds=True)
    hp = (5.0, 0.03, 0.02, 1e-3, 3, 2)
    sop = rowblock.slot_order(500)
    want = cpu_oracle.relaxed_optimize_layout(*args, 400, *hp, seed=1, slot_of_point=sop, trace=True)
    got = _lib.fit(*args, 400, *hp, mode=_lib.MODE_ROWBLOCK, seed=1, trace=True)
    assert want["converged"] and want["iterations_run"] < 400
    assert got["converged"]
    assert abs(got["iterations_run"] - want["iterations_run"]) <= 6      # a plateau test at 1e-3 may flip one check later
    k = min(got["iterations_run"], want["iterations_run"])
    a, b = got["trace_mae"][:k], want["trace_mae"][:k]
    assert np.array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_allclose(a[~np.isnan(a)], b[~np.isnan(b)], rtol=2e-3)
    assert got["final_mae"] == pytest.approx(want["final_mae"], rel=2e-3)


# ------------------------------------------------------------------ sharding ---------------------
@pytest.mark.parametrize("n,d,ranks", [(2300, 32, (2, 4)), (1000, 19, (3,))])
def test_rowblock_highdim_result_does_not_depend_on_the_number_of_ranks(n, d, ranks):
    args = small_problem(n, d, 0.05, n + d, thresholds=True)
    hp = (5.0, 0.02, 0.02, 1e-3, 3, 2)
    one = _lib.fit(*args, 40, *hp, mode=_lib.MODE_ROWBLOCK, seed=9, trace=True)
    for r in ranks:
        ls = rowblock.LocalShards(*args, 40, *hp, n_ranks=r, seed=9)
        try:
            ls.run(40)
            for q in {0, r - 1}:
                got = ls.result(rank=q, trace=True)
                assert np.array_equal(got["positions"], one["positions"]), (r, q)
                assert (got["final_mae"], got["iterations"], got["iterations_run"], got["converged"], got["pair_updates"]) == \
                       (one["final_mae"], one["iterations"], one["iterations_run"], one["converged"], one["pair_updates"])
                assert np.array_equal(got["trace_mae"], one["trace_mae"], equal_nan=True)
            info = ls.shards[0].info()
            stride = (d + 3) // 4 * 4
            assert info["n_ranks"] == r and info["ndim"] == d and info["stride"] == stride
            assert info["peer_store_bytes_per_iteration"] == (r - 1) * info["own_rows"] * stride * 4
        finally:
            ls.close()


# ------------------------------------------------------------------ hold-out, interrupt ----------
def test_rowblock_highdim_holdout_and_interrupt():
    init, deg, ei, ej, ed, et = small_problem(400, 24, 0.2, 5, thresholds=False)
    held = np.random.default_rng(0).random(len(ei)) < 0.1
    g = _lib.fit(init, deg, ei[~held], ej[~held], ed[~held], et[~held], 30, *HP, mode=_lib.MODE_ROWBLOCK,
                 holdout=(ei[held], ej[held], ed[held]))
    dist = np.linalg.norm(g["positions"][ei[held]] - g["positions"][ej[held]], axis=1)
    assert g["holdout_count"] == held.sum()
    assert g["holdout_sum_abs"] == pytest.approx(np.abs(ed[held] - dist).sum(), rel=1e-9)
    calls = []
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(init, deg, ei, ej, ed, et, 500, *HP[:3], 1e-12, 1000, 3, mode=_lib.MODE_ROWBLOCK,
                 interrupt=lambda: (calls.append(1), len(calls) > 2)[1])
    assert e.value.status == _lib.ERR_INTERRUPTED and len(calls) == 3


# ------------------------------------------------------------------ statistics --------------------
def _parity(gpu, cpu, rel):
    gpu, cpu = np.asarray(gpu), np.asarray(cpu)
    se = np.sqrt(gpu.var(ddof=1) / len(gpu) + cpu.var(ddof=1) / len(cpu))
    assert abs(gpu.mean() - cpu.mean()) <= max(2 * se, rel * cpu.mean()), (gpu.mean(), cpu.mean(), se, gpu, cpu)


@pytest.mark.parametrize("d", [20, 32])
def test_rowblock_highdim_statistical_parity_with_the_reference_loop(d):
    """Edge MAE at the best state, held-out MAE and distance-reconstruction error of fits that never saw 10 % of the exact
    cells: row-block mode vs the reference's std::shuffle loop, 10 seeds, thresholds on."""
    n = 400
    mae, hold, rec = ([], []), ([], []), ([], [])
    for seed in range(10):
        init, deg, ei, ej, ed, et = small_problem(n, d, 0.12, 5000 + 100 * d + seed, thresholds=True)
        rng = np.random.default_rng(seed)
        held = (rng.random(len(ei)) < 0.1) & (et == 0)
        tr = ~held
        deg_tr = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
        train = (init, deg_tr, ei[tr], ej[tr], ed[tr], et[tr])
        g = _lib.fit(*train, 200, *HP, mode=_lib.MODE_ROWBLOCK, seed=seed)
        c = cpu_oracle.optimize_layout_exact(*train, 200, *HP, seed=seed)
        for k, r in enumerate((g, c)):
            dist = np.linalg.norm(r["positions"][ei] - r["positions"][ej], axis=1)
            mae[k].append(r["final_mae"])
            hold[k].append(np.abs(ed[held] - dist[held]).mean())
            rec[k].append(np.abs(ed[et == 0] - dist[et == 0]).mean())
    _parity(mae[0], mae[1], 0.03)
    _parity(hold[0], hold[1], 0.03)
    _parity(rec[0], rec[1], 0.03)


# ------------------------------------------------------------------ form and errors ---------------
def test_rowblock_highdim_runs_the_fp32_difference_form(monkeypatch):
    monkeypatch.delenv("TOPOLOW_REP_VARIANT", raising=False)
    args = small_problem(600, 20, 0.08, 31, thresholds=True)
    sh = rowblock.Shard(*args, 4, *HP, seed=3)
    try:
        sh.run(4)
        info = sh.info()
        assert sh.result()["iterations_run"] == 4
    finally:
        sh.close()
    assert info["repulsion_form"] == 5 and info["tensor_form_iterations"] == -1, info
    assert info["ndim"] == 20 and info["stride"] == 20


def test_rowblock_highdim_rejects_other_forms_and_ndim_over_32(monkeypatch):
    args = small_problem(600, 20, 0.08, 31, thresholds=True)
    monkeypatch.setenv("TOPOLOW_REP_VARIANT", "11")
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(*args, 4, *HP, mode=_lib.MODE_ROWBLOCK)
    assert e.value.status == _lib.ERR_BAD_ARG
    with pytest.raises(_lib.TopolowError) as e:
        rowblock.Shard(*args, 4, *HP)
    assert e.value.status == _lib.ERR_BAD_ARG
    monkeypatch.setenv("TOPOLOW_REP_VARIANT", "5")
    assert _lib.fit(*args, 4, *HP, mode=_lib.MODE_ROWBLOCK)["iterations_run"] == 4
    monkeypatch.delenv("TOPOLOW_REP_VARIANT")
    wide = small_problem(300, 33, 0.1, 7, thresholds=True)
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(*wide, 4, *HP, mode=_lib.MODE_ROWBLOCK)
    assert e.value.status == _lib.ERR_BAD_ARG and "replay mode takes any ndim" in str(e.value)


# ------------------------------------------------------------------ end to end --------------------
def test_rowblock_highdim_end_to_end():
    rng = np.random.default_rng(11)
    n = 300
    X = rng.normal(size=(n, 20)) * 2
    D = np.linalg.norm(X[:, None] - X[None], axis=2)
    mask = np.triu(rng.random((n, n)) < 0.7, 1)
    M = np.where(mask | mask.T, D, np.nan)
    np.fill_diagonal(M, 0.0)
    r = core.euclidean_embedding(M, 20, 60, k0=5.0, cooling_rate=0.01, c_repulsion=0.02, mode="rowblock", seed=2)
    assert r.positions.shape == (n, 20) and np.all(np.isfinite(r.positions))
    assert r.est_distances.shape == (n, n) and np.isfinite(r.mae)
    assert r.iter >= 0 and r.parameters["ndim"] == 20 and np.isfinite(r.convergence["error"])
    iu = np.nonzero(np.triu(mask, 1))
    c = core.euclidean_embedding_coo(n, iu[0], iu[1], D[iu], 24, 60, k0=5.0, cooling_rate=0.01, c_repulsion=0.02,
                                     mode="rowblock", seed=2)
    assert c.positions.shape == (n, 24) and np.all(np.isfinite(c.positions))
    assert len(c.est_distances) == len(iu[0]) and np.isfinite(c.mae)
