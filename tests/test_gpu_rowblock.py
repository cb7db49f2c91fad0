"""GPU parity tests of the row-block ("relaxed", owner-computes) mode - topolow_b200/csrc/rowblock.cu,
the scheme SURVEY.md section 8e names for one large map across GPUs.  Everything goes through the C ABI.

Bars:
  numerics     FP32 kernels vs the FP64 CPU restatement of the same scheme (oracle/relaxed_oracle.cpp) on the
               same visiting order: 99 % of the coordinates within 2e-4 of the coordinate scale, all within
               2e-3, after 6 iterations; edge MAE within 1e-3 relative
  sharding     the result is bit-identical for 1, 2, 3 ranks (lock-step emulation of the ranks on one GPU; with
               two GPUs also as two processes over CUDA IPC)
  statistics   vs the REFERENCE's sequential random-shuffle loop (oracle/topolow_oracle.cpp), 10 seeds, same
               inputs: edge MAE, held-out MAE and distance-reconstruction error agree within
               max(2 x SE of the difference, 3 %) - on synthetic data and on BASELINE.json configs[0] / [1]
               (H3N2, HIV with thresholds, ndim 5, published hyper-parameters)
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_fixture, small_problem
from oracle import cpu_oracle
from tools import synth
from topolow_b200 import _lib, rowblock

pytestmark = pytest.mark.gpu

HP = (5.0, 0.01, 0.02, 1e-4, 5, 3)


def _gpu_count():
    import torch
    return torch.cuda.device_count()


# ------------------------------------------------------------------ numerics ---------------------
@pytest.mark.parametrize("n,d,dens", [(300, 2, 0.2), (700, 5, 0.1), (520, 3, 0.15), (600, 10, 0.08), (2100, 16, 0.02),
                                      (400, 7, 0.3), (257, 2, 0.2)])
def test_rowblock_tracks_its_fp64_restatement(n, d, dens):
    args = small_problem(n, d, dens, 10 * n + d, thresholds=True)
    sop = rowblock.slot_order(n)
    want = cpu_oracle.relaxed_optimize_layout(*args, 6, *HP, seed=4, slot_of_point=sop)
    got = _lib.fit(*args, 6, *HP, mode=_lib.MODE_ROWBLOCK, seed=4)
    scale = max(np.abs(want["positions"]).max(), 1.0)
    err = np.abs(got["positions"] - want["positions"])
    assert np.quantile(err, 0.99) <= 2e-4 * scale and err.max() <= 2e-3 * scale, (np.quantile(err, 0.99), err.max(), scale)
    assert got["final_mae"] == pytest.approx(want["final_mae"], rel=1e-3)
    assert got["iterations"] == want["iterations"] and got["iterations_run"] == 6
    assert got["final_k"] == pytest.approx(want["final_k"], rel=1e-12)
    assert got["pair_updates"] == 6 * n * (n - 1) // 2


def test_rowblock_controller_and_trace_follow_the_restatement():
    # early stop: the same check iterations, the same best iteration, MAE trace within FP32 noise
    args = small_problem(500, 3, 0.2, 77, thresholds=True)
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


def test_rowblock_holdout_trace_and_interrupt():
    init, deg, ei, ej, ed, et = small_problem(400, 4, 0.2, 5, thresholds=False)
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


def test_rowblock_error_paths(monkeypatch):
    init = np.zeros((300, 2)); init[:, 0] = np.arange(300)
    deg = np.full(300, 2, dtype=np.int32)
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(init, deg, [0], [1], [1.0], [0], 20, 1e30, 0.01, 1e38, convergence_window=100, convergence_check_freq=50,
                 mode=_lib.MODE_ROWBLOCK)
    assert e.value.status == _lib.ERR_NONFINITE
    assert "Numerical instability at iteration 10. Reduce k0 or c_repulsion." in str(e.value)
    args = list(small_problem(300, 2, 0.1, 0))
    bad = list(args); bad[2] = np.array(args[2]); bad[2][0] = 999
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(*bad, 5, 1.0, 0.01, 0.01, mode=_lib.MODE_ROWBLOCK)
    assert e.value.status == _lib.ERR_BAD_ARG and "edge index" in str(e.value)
    with pytest.raises(_lib.TopolowError) as e:
        rowblock.LocalShards(*args, 5, 1.0, 0.01, 0.01, n_ranks=3)      # 300 points = 2 row tiles
    assert e.value.status == _lib.ERR_BAD_ARG and "too few points" in str(e.value)
    dup = [args[0], args[1]] + [np.r_[a, a[:5]] for a in args[2:]]      # a pair listed twice is tolerated
    r = _lib.fit(*dup, 5, 1.0, 0.01, 0.01, mode=_lib.MODE_ROWBLOCK)
    assert np.all(np.isfinite(r["positions"]))
    args8 = small_problem(600, 8, 0.08, 8)
    for form in ("6", "10"):                                          # forms that were measured and dropped
        monkeypatch.setenv("TOPOLOW_REP_VARIANT", form)
        with pytest.raises(_lib.TopolowError) as e:
            _lib.fit(*args8, 4, 1.0, 0.01, 0.01, mode=_lib.MODE_ROWBLOCK)
        assert e.value.status == _lib.ERR_BAD_ARG and "takes 5" in str(e.value)


# ------------------------------------------------------------------ sharding ---------------------
@pytest.mark.parametrize("n,d,ranks", [(1000, 3, (2, 3)), (2300, 16, (2, 4)), (1500, 5, (5,))])
def test_rowblock_result_does_not_depend_on_the_number_of_ranks(n, d, ranks):
    args = small_problem(n, d, 0.05, n + d, thresholds=True)
    hp = (5.0, 0.02, 0.02, 1e-3, 3, 2)
    one = _lib.fit(*args, 40, *hp, mode=_lib.MODE_ROWBLOCK, seed=9, trace=True)
    for r in ranks:
        ls = rowblock.LocalShards(*args, 40, *hp, n_ranks=r, seed=9)
        ls.run(40)
        for q in {0, r - 1}:
            got = ls.result(rank=q, trace=True)
            assert np.array_equal(got["positions"], one["positions"]), (r, q)
            assert (got["final_mae"], got["iterations"], got["iterations_run"], got["converged"]) == \
                   (one["final_mae"], one["iterations"], one["iterations_run"], one["converged"])
            assert np.array_equal(got["trace_mae"], one["trace_mae"], equal_nan=True)
        info = ls.shards[0].info()
        assert info["n_ranks"] == r and info["peer_store_bytes_per_iteration"] == (r - 1) * info["own_rows"] * info["stride"] * 4
        ls.close()


def test_rowblock_stepping_in_pieces_equals_one_run():
    args = small_problem(900, 4, 0.05, 3, thresholds=True)
    one = _lib.fit(*args, 25, *HP, mode=_lib.MODE_ROWBLOCK, seed=2)
    sh = rowblock.Shard(*args, 25, *HP, seed=2)
    for k in (1, 7, 3, 20):      # asks for more than n_iter in total: clamped
        sh.run(k)
    got = sh.result()
    sh.close()
    assert np.array_equal(got["positions"], one["positions"]) and got["iterations_run"] == 25


@pytest.mark.skipif("_gpu_count() < 2")
def test_rowblock_two_processes_over_cuda_ipc_equal_one_rank(tmp_path):
    outs = []
    for world in (1, 2):
        out = str(tmp_path / f"ranks{world}.npz")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
               "127.0.0.1", "--master-port", str(29531 + world), os.path.join(ROOT, "tools", "gpu_rowblock_ranks.py"),
               "--points", "3000", "--ndim", "5", "--iters", "12", "--out", out]
        subprocess.run(cmd, check=True, timeout=600, cwd=ROOT)
        outs.append(np.load(out))
    assert np.array_equal(outs[0]["positions"], outs[1]["positions"])
    assert float(outs[0]["final_mae"]) == float(outs[1]["final_mae"])


@pytest.mark.skipif("_gpu_count() < 2")
def test_rowblock_two_devices_in_one_process_equal_one_rank():
    args = small_problem(1200, 5, 0.05, 8, thresholds=True)
    one = _lib.fit(*args, 20, *HP, mode=_lib.MODE_ROWBLOCK, seed=9)
    ls = rowblock.LocalShards(*args, 20, *HP, n_ranks=2, devices=[0, 1], seed=9)
    ls.run(20)
    got = ls.result(rank=1)
    ls.close()
    assert np.array_equal(got["positions"], one["positions"])


# ------------------------------------------------------------------ statistics --------------------
def _parity(gpu, cpu, rel):
    gpu, cpu = np.asarray(gpu), np.asarray(cpu)
    se = np.sqrt(gpu.var(ddof=1) / len(gpu) + cpu.var(ddof=1) / len(cpu))
    assert abs(gpu.mean() - cpu.mean()) <= max(2 * se, rel * cpu.mean()), (gpu.mean(), cpu.mean(), se, gpu, cpu)


def test_rowblock_statistical_parity_with_the_reference_loop():
    """Edge MAE at the best state, held-out MAE and distance-reconstruction error of fits that never saw 10 % of
    the cells: row-block mode vs the reference's std::shuffle loop, 10 seeds, thresholds on."""
    n, d = 400, 3
    mae, hold, rec = ([], []), ([], []), ([], [])
    for seed in range(10):
        init, deg, ei, ej, ed, et = small_problem(n, d, 0.12, 3000 + seed, thresholds=True)
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


PUBLISHED = {   # inst/examples/methods-comparison-h3n2-hiv-denv.Rmd:312-331 (k0, cooling_rate, c_repulsion), ndim 5
    "h3n2": (14.76214, 0.03641074, 0.002943064),
    "hiv": (3.550036, 0.04130713, 0.0007038619),
}


@pytest.mark.parametrize("name", ["h3n2", "hiv"])
def test_rowblock_parity_on_the_bundled_maps(name):
    """BASELINE.json configs[0] / configs[1]: the bundled H3N2 and HIV tables (HIV with '>' thresholds), ndim 5,
    mapping_max_iter 1000, published hyper-parameters; 10 % of the exact cells held out; 10 seeds."""
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
        g = _lib.fit(*train, mode=_lib.MODE_ROWBLOCK, seed=seed)
        c = cpu_oracle.optimize_layout_exact(*train, seed=seed)
        for k, r in enumerate((g, c)):
            dist = np.linalg.norm(r["positions"][ei] - r["positions"][ej], axis=1)
            mae[k].append(r["final_mae"])
            hold[k].append(np.abs(ed[held] - dist[held]).mean())
    _parity(mae[0], mae[1], 0.03)
    _parity(hold[0], hold[1], 0.03)


def test_rowblock_cfg3_size_against_the_reference_loop():
    """BASELINE.json configs[2] shape at a size the dense CPU loop finishes in a minute: 3000 points, 95 % missing,
    ndim 10, thresholds, 60 iterations, 3 seeds of the shuffle: edge MAE and held-out MAE within 3 %."""
    n, d = 3000, 10
    prob = synth.make_problem(n, d, 0.95, seed=1)
    ei, ej, ed, et = prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"]
    held = (np.random.default_rng(5).random(len(ei)) < 0.1) & (et == 0)
    tr = ~held
    deg_tr = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
    train = (prob["initial_positions"], deg_tr, ei[tr], ej[tr], ed[tr], et[tr], 60, 5.0, 0.01, 0.02, 1e-4, 100, 3)
    g = _lib.fit(*train, mode=_lib.MODE_ROWBLOCK, seed=0)
    gd = np.linalg.norm(g["positions"][ei] - g["positions"][ej], axis=1)
    cm, ch = [], []
    for seed in range(3):
        c = cpu_oracle.optimize_layout_exact(*train, seed=seed)
        cd = np.linalg.norm(c["positions"][ei] - c["positions"][ej], axis=1)
        cm.append(c["final_mae"]); ch.append(np.abs(ed[held] - cd[held]).mean())
    assert g["final_mae"] == pytest.approx(np.mean(cm), rel=0.03), (g["final_mae"], cm)
    assert np.abs(ed[held] - gd[held]).mean() == pytest.approx(np.mean(ch), rel=0.03), (ch,)


# ------------------------------------------------------------------ the forms of the repulsion pass ----
def test_rowblock_repulsion_forms_agree_and_the_device_picks_one_per_iteration(monkeypatch):
    """The forms of the repulsion pass - FP32 difference form (TOPOLOW_REP_VARIANT=5), two-GEMM tcgen05 form with the
    weights by square root + reciprocal (11, TOPOLOW_TC_SERIES=0) or by the one-MUFU series (11, TOPOLOW_TC_SERIES=1) -
    compute the same sums: after 8 iterations each is where the FP32 form is, within the TF32 noise (99 % of the
    coordinates within 2e-3 of the map's scale, all within 2e-2, MAE 1 %).  The policy's run (no variable set) chooses among them per iteration on the
    device and reports how many iterations ran a tensor form.  (Kept last in the file on purpose.)"""
    n, d, iters = 1500, 8, 8
    args = small_problem(n, d, 0.05, 4242, thresholds=True)
    runs = {}
    for name, env in (("f32", {"TOPOLOW_REP_VARIANT": "5"}),
                      ("tensor", {"TOPOLOW_REP_VARIANT": "11", "TOPOLOW_TC_SERIES": "0"}),
                      ("series", {"TOPOLOW_REP_VARIANT": "11", "TOPOLOW_TC_SERIES": "1"}),
                      ("policy", {})):
        for k in ("TOPOLOW_REP_VARIANT", "TOPOLOW_TC_SERIES", "TOPOLOW_ADAPTIVE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        sh = rowblock.Shard(*args, iters, *HP, seed=3)
        try:
            sh.run(iters)
            runs[name] = (sh.result(), sh.info())
        finally:
            sh.close()
    base = runs["f32"][0]
    scale = max(np.abs(base["positions"]).max(), 1.0)
    for name in ("tensor", "series", "policy"):
        r = runs[name][0]
        err = np.abs(r["positions"] - base["positions"])
        # TF32 weights (truncated: 2.4e-4 low on average) and TF32 partner coordinates act on moves of the order of the map
        # itself while the start line unfolds, which the forced tensor forms - unlike the policy - take from iteration 0
        assert np.quantile(err, 0.99) <= 2e-3 * scale and err.max() <= 2e-2 * scale, (name, np.quantile(err, 0.99), err.max(), scale)
        assert r["final_mae"] == pytest.approx(base["final_mae"], rel=1e-2), name
        assert r["iterations_run"] == iters
    assert runs["f32"][1]["repulsion_form"] == 5 and runs["f32"][1]["tensor_form_iterations"] == -1
    assert runs["series"][1]["repulsion_form"] == 11 and runs["series"][1]["tensor_form_iterations"] == -1
    info = runs["policy"][1]
    assert info["repulsion_form"] == 11 and 0 <= info["tensor_form_iterations"] <= iters, info
