"""CPU tests of the host side: C-ABI surface, schedule coverage, the Python mirror of the R glue
(against oracle/r_glue.py), fold construction, sharding over ranks (gloo, world size 2)."""
import ctypes as C
import json
import math
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

from conftest import ROOT, has_cuda, random_r_matrix, small_problem
from oracle import r_glue
from topolow_b200 import _lib, core, cv, shard


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "topolow_b200.h")).read()
    declared = set(re.findall(r"TOPOLOW_API\s+[\w\s\*]+?\b(topolow_\w+)\s*\(", header))
    assert declared == set(_lib.EXPORTS)
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (topolow_\w+)", nm))
    assert declared <= exported
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name)
    assert b"sm_100a" in L.topolow_version()
    sizes = (C.c_int64 * 3)()
    L.topolow_abi_sizes(C.byref(sizes))       # the ctypes mirror of the three structs matches the header
    assert list(sizes) == [C.sizeof(_lib.Problem), C.sizeof(_lib.Params), C.sizeof(_lib.Result)]


@pytest.mark.skipif(has_cuda(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_without_a_device():
    args = small_problem(20, 2, 0.5, 0)
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit(*args, 5, 1.0, 0.01, 0.01)
    assert e.value.status == _lib.ERR_CUDA
    with pytest.raises(_lib.TopolowError):
        _lib.est_distances(np.zeros((4, 2)))


def test_too_few_points_status():
    L = _lib.lib()
    pa = _lib.ProblemArrays(np.zeros((1, 2)), [1], [], [], [], [])
    pr, _ = _lib.make_params(5, 1.0, 0.01, 0.01)
    out = np.zeros((1, 2))
    res = _lib.Result()
    res.positions = out.ctypes.data_as(_lib._dp)
    import ctypes as C
    rc = L.topolow_fit(C.byref(pa.struct), C.byref(pr), C.byref(res))
    assert rc == _lib.ERR_TOO_FEW_POINTS
    assert res.message.decode() == "Need at least 2 points for embedding"   # src/optimization.cpp:131


@pytest.mark.parametrize("n", [2, 3, 31, 33, 65, 97, 193, 335, 700, 1025, 1500])
@pytest.mark.parametrize("prec", [_lib.PREC_F32, _lib.PREC_F64_EXACT])
@pytest.mark.parametrize("tile_points", [32, 64, 96])
def test_schedule_visits_every_pair_exactly_once(n, prec, tile_points):
    for it, max_ctas in ((0, 0), (7, 3)):
        order, geo = _lib.schedule_enumerate(n, 5, it, precision=prec, seed=n + it, max_ctas=max_ctas,
                                             tile_points=tile_points)
        a = np.minimum(order[:, 0], order[:, 1]).astype(np.int64)
        b = np.maximum(order[:, 0], order[:, 1]).astype(np.int64)
        assert (a != b).all() and a.min() >= 0 and b.max() < n
        assert len(np.unique(a * n + b)) == n * (n - 1) // 2
        assert geo["super_blocks"] == 2 * geo["ctas"] * geo["tasks_per_cta"]
        assert geo["super_blocks"] * geo["warps_per_cta"] >= geo["tiles"]


def test_schedule_steps_are_matchings_and_orders_differ_between_iterations():
    n = 200
    o0, _ = _lib.schedule_enumerate(n, 3, 0, seed=1)
    o1, _ = _lib.schedule_enumerate(n, 3, 1, seed=1)
    assert not np.array_equal(o0, o1)
    # the enumerator emits one ring / xor step of one tile pair at a time: consecutive pairs sharing
    # a tile pair and step never repeat a point.  Check greedily: a run of pairs with all-distinct points
    # must on average be long (>= 8) - a sequential-only order would give runs of ~ sqrt(n).
    runs, seen, cur = [], set(), 0
    for i, j in o0:
        if i in seen or j in seen:
            runs.append(cur); seen, cur = set(), 0
        seen.update((int(i), int(j))); cur += 1
    assert np.mean(runs) >= 8


VALIDATION = [
    (dict(ndim=-1), "ndim must be a positive integer"),
    (dict(k0=-1), "k0 must be a positive number"),
    (dict(cooling_rate=1.5), "cooling_rate must be between 0 and 1"),
    (dict(c_repulsion=0), "c_repulsion must be a positive number"),
    (dict(relative_epsilon=-1), "relative_epsilon must be a positive number"),
    (dict(convergence_counter=0.5), "convergence_counter must be a positive integer"),
    (dict(mapping_max_iter=0), "mapping_max_iter must be a positive integer"),
    (dict(convergence_check_freq=0), "convergence_check_freq must be a positive integer"),
]


@pytest.mark.parametrize("override,msg", VALIDATION)
def test_validation_messages_match_the_reference(override, msg):
    # tests/testthat/test-core.R:22-65, R/core.R:202-264
    m = np.array(random_r_matrix(4, 1.0, 0, thresholds=False), dtype=float)
    kw = dict(ndim=2, mapping_max_iter=10, k0=1.0, cooling_rate=0.01, c_repulsion=0.01, relative_epsilon=1e-4,
              convergence_counter=5)
    kw.update(override)
    with pytest.raises(ValueError, match=re.escape(msg)):
        core.euclidean_embedding(m, **kw)


def test_matrix_validation_and_k0_warning():
    with pytest.raises(ValueError, match="dissimilarity_matrix must be a matrix"):
        core.euclidean_embedding("not a matrix", 2, 10, 1.0, 0.01, 0.01)
    with pytest.raises(ValueError, match="dissimilarity_matrix must be square"):
        core.euclidean_embedding(np.arange(6.0).reshape(2, 3), 2, 10, 1.0, 0.01, 0.01)
    m = np.array(random_r_matrix(4, 1.0, 0, thresholds=False), dtype=float)
    with pytest.raises(ValueError, match="initial_positions must have same number of rows"):
        core.euclidean_embedding(m, 2, 10, 1.0, 0.01, 0.01, initial_positions=np.zeros((5, 2)))
    with pytest.raises(ValueError, match="initial_positions must have ndim columns"):
        core.euclidean_embedding(m, 2, 10, 1.0, 0.01, 0.01, initial_positions=np.zeros((4, 3)))
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        try:
            core.euclidean_embedding(m, 2, 10, 35.0, 0.01, 0.01)
        except _lib.TopolowError:
            pass  # no GPU here: the warning fires before the native call
        assert any("High k0 value" in str(x.message) for x in w)


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("preserve", [True, False])
def test_build_problem_matches_the_r_glue_restatement(seed, preserve):
    m = random_r_matrix(23, 0.4, seed)
    got = core.build_problem(m, preserve)
    want = r_glue.prepare(m, preserve)
    assert (got["order"] is None) == (want["order"] is None)
    if got["order"] is not None:
        assert np.array_equal(got["order"], want["order"])
    for k in ("degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh"):
        assert np.array_equal(got[k], want[k]), k


def test_parse_numeric_and_character_matrices_agree():
    m = random_r_matrix(12, 0.6, 9, thresholds=False)
    num = np.array([[np.nan if x is None else float(x) for x in row] for row in m])
    a, b = core.build_problem(m, True), core.build_problem(num, True)
    for k in ("degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh"):
        assert np.array_equal(a[k], b[k])


def test_folds_follow_the_reference_scheme():
    # R/adaptive_sampling.R:2568-2598
    m = random_r_matrix(20, 0.6, 4)
    folds_a = cv.make_folds(m, 5, np.random.default_rng(7))
    folds_b = r_glue.make_folds(m, 5, np.random.default_rng(7))
    assert len(folds_a) == len(folds_b) == 5
    for a, b in zip(folds_a, folds_b):
        assert np.array_equal(a, b)
    non_na = sum(x is not None for x in m.ravel())
    assert all(len(f) == non_na // 10 for f in folds_a)
    seen = set()
    for f in folds_a:            # a cell and its mirror leave the pool together (a single draw may
        cells = {(int(i) % 20, int(i) // 20) for i in f}   # still hold both orientations of a pair)
        assert not (cells & seen)
        seen |= cells | {(c, r) for r, c in cells}


def test_error_calculator_matches_oracle_and_reference_kats():
    rng = np.random.default_rng(0)
    true = random_r_matrix(9, 0.8, 2)
    inp = true.copy()
    inp[1, 4] = inp[4, 1] = None
    inp[0, 0] = None
    pred = rng.uniform(0, 5, size=(9, 9))
    got = cv.error_calculator_comparison(pred, true, inp)
    want = r_glue.error_calculator_comparison(pred, true, inp)
    for k in ("InSampleError", "OutSampleError", "InSamplePercentageError", "OutSamplePercentageError"):
        np.testing.assert_array_equal(got["report_df"][k], want[k])
    assert got["Completeness"] == want["Completeness"]
    # tests/testthat/test-diagnostics.R:5-20
    t3 = np.array([[0, 1, 2], [1, 0, 3], [2, 3, 0]], dtype=float)
    i3 = t3.copy(); i3[0, 2] = i3[2, 0] = np.nan
    e = cv.error_calculator_comparison(t3 + 0.1, t3, i3)["report_df"]
    assert np.sum(~np.isnan(e["OutSampleError"])) == 2 and np.sum(~np.isnan(e["InSampleError"])) == 7
    with pytest.raises(ValueError, match="All matrices must have the same dimensions"):
        cv.error_calculator_comparison(np.zeros((2, 2)), t3)


def test_partition_is_longest_first_and_complete():
    costs = [5, 1, 9, 3, 3, 7, 2]
    parts = shard.partition(costs, 3)
    assert sorted(j for p in parts for j in p) == list(range(7))
    loads = [sum(costs[j] for j in p) for p in parts]
    assert max(loads) - min(loads) <= max(costs)
    assert shard.partition(costs, 1) == [[2, 5, 0, 3, 4, 6, 1]]


_GLOO_SCRIPT = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch.distributed as dist
from topolow_b200 import shard
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
jobs = [dict(degrees=np.ones(n, np.int32), n_iter=it, tag=i) for i, (n, it) in enumerate([(50, 10), (20, 5), (80, 3), (10, 100), (60, 7)])]
calls = []
def fake_batch(js, device=0):            # stands in for _lib.fit_batch: no GPU on this box
    calls.append(len(js))
    return [dict(status=0, tag=j["tag"], rank=dist.get_rank()) for j in js]
out = shard.run_sharded(jobs, fit_batch=fake_batch)
assert [r["tag"] for r in out] == [0, 1, 2, 3, 4], out
assert len(calls) == 1                      # one batch call per rank
assert {{r["rank"] for r in out}} == {{0, 1}}
parts = shard.partition([shard.job_cost(j) for j in jobs], 2)
assert all(out[j]["rank"] == r for r, p in enumerate(parts) for j in p)
dist.barrier(); dist.destroy_process_group()
print("ok")
"""


def test_sharding_across_two_ranks_with_gloo(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "gloo_shard.py"
    script.write_text(_GLOO_SCRIPT.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=120)
        assert p.returncode == 0, err[-2000:]
        assert "ok" in out


def test_likelihood_batch_holdout_cells_follow_the_reordering(monkeypatch):
    """likelihood_batch hands every fit its hold-out cells in the row numbering of the fold's training
    problem (which euclidean_embedding-style reordering permutes unless preserve_order).  A stub "fit"
    that returns its initial positions makes the expected residuals computable by hand."""
    m = random_r_matrix(30, 0.6, 11)
    value, code, is_na = core.parse_dissimilarity(m)
    folds = cv.make_folds(m, 3, np.random.default_rng(2))
    G = np.random.default_rng(5).normal(size=(30, 2)) * 4          # "embedding" in the caller's row numbering

    def stub_fit_batch(jobs, device=0):
        out = []
        for j in jobs:
            pos = np.asarray(j["initial_positions"], dtype=float)
            hi, hj, ht = j["holdout"]
            ok = ~np.isnan(ht)
            d = np.linalg.norm(pos[hi] - pos[hj], axis=1)
            out.append(dict(status=_lib.OK, positions=pos, holdout_sum_abs=float(np.abs(ht[ok] - d[ok]).sum()),
                            holdout_count=int(ok.sum()), iterations=1, converged=True))
        return out

    monkeypatch.setattr(_lib, "fit_batch", stub_fit_batch)
    for preserve in (True, False):
        inits, want = [], []
        for h in folds:
            prob, ci, cj, tr = cv._fold_job(value, code, is_na, np.asarray(h), preserve)
            inits.append(G if prob["order"] is None else G[prob["order"]])
            want.append(np.abs(tr - np.linalg.norm(G[ci] - G[cj], axis=1)).mean())
        assert preserve or any(cv._fold_job(value, code, is_na, np.asarray(h), False)[0]["order"] is not None for h in folds)
        got = cv.likelihood_batch(m, [dict(N=2, k0=1.0, cooling_rate=0.01, c_repulsion=0.01)], 5, 1e-4, folds=3,
                                  preserve_order=preserve, fold_indices=folds, init_list=[inits])
        assert [f["Holdout_MAE"] for f in got[0]["folds"]] == pytest.approx(want, rel=1e-12)


# ------------------------------------------------------------------ the .Call shim ---------------
@pytest.fixture(scope="module")
def shim_cpu(tmp_path_factory):
    from conftest import build_r_shim_harness
    return build_r_shim_harness(str(tmp_path_factory.mktemp("shim") / "harness_cpu"), real_library=False)


def _harness(exe, *args):
    out = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


def _clean(r):
    assert r["protect_depth"] == 0 and r["type_errors"] == 0 and r["rng_violations"] == 0 and r["rng_open"] == 0
    assert r["raw_interrupt_jumps"] == 0


def test_r_shim_registers_both_entries(shim_cpu):
    r = _harness(shim_cpu, "register")
    assert r["routines"] == {"_topolow_optimize_layout_b200": 16, "_topolow_fit_batch_b200": 3}    # src/RcppExports.cpp:41-49
    assert r["dynamic_symbols"] == 0


def test_r_shim_single_call_marshals_every_field(shim_cpu, tmp_path):
    from conftest import write_problem_bin
    init, deg, ei, ej, ed, et = small_problem(40, 3, 0.3, 1)
    write_problem_bin(tmp_path / "p.bin", init, deg, ei, ej, ed, et)
    r = _harness(shim_cpu, "single", tmp_path / "p.bin", tmp_path / "o.bin", 100, 5.0, 0.01, 0.02, 1e-4, 5, 3, "rowblock")
    _clean(r)
    assert r["names"] == ["positions", "converged", "iterations", "final_mae", "final_k"]      # src/optimization.cpp:375-381
    assert r["types"] == [14, 10, 13, 14, 14] and r["dim"] == [40, 3]                          # REALSXP, LGLSXP, INTSXP, REALSXP x 2
    out = np.fromfile(tmp_path / "o.bin")
    # the recording fake answers with functions of what it was handed (integration/r_stub/fake_topolow.c)
    assert out[0] == 1 and out[1] == 100 - 3
    assert out[2] == pytest.approx(float(np.sum(ed * (1 + et) + ei - ej)), rel=1e-12)
    assert out[3] == pytest.approx(5.0 * 0.99 + 0.02 + 1e-4, rel=1e-15)
    pos = out[4:].reshape(3, 40).T
    np.testing.assert_allclose(pos, 2 * init + deg[:, None], rtol=0, atol=0)
    # a second scenario in the default mode: seed drawn inside GetRNGstate / PutRNGstate (two draws of the fixed stream)
    r2 = _harness(shim_cpu, "single", tmp_path / "p.bin", tmp_path / "o2.bin", 50, 1.0, 0.5, 0.0, 0.0, 4, 1)
    _clean(r2)
    assert np.fromfile(tmp_path / "o2.bin")[0] == 0          # convergence_window reached the library as 4


def test_r_shim_errors_and_interrupts_leave_through_the_shim(shim_cpu, tmp_path):
    from conftest import write_problem_bin
    r = _harness(shim_cpu, "too_few")
    assert r["left_by"] == "Rf_error" and r["message"] == "Need at least 2 points for embedding"   # src/optimization.cpp:131
    _clean(r)
    write_problem_bin(tmp_path / "p.bin", *small_problem(30, 2, 0.3, 2))
    r = _harness(shim_cpu, "interrupt", tmp_path / "p.bin", 3)
    # the interrupt is caught inside R_ToplevelExec, reported to the library as a return value, and only after the
    # library has returned TOPOLOW_ERR_INTERRUPTED does the shim raise the R condition - never a jump through it
    assert r["left_by"] == "Rf_onintr" and r["onintr_calls"] == 1 and r["interrupt_checks"] == 3
    _clean(r)
    r = _harness(shim_cpu, "interrupt", tmp_path / "p.bin", 0)      # no interrupt: polled between chunks, returns normally
    assert r["left_by"] == "return" and r["interrupt_checks"] == 4
    _clean(r)


def test_r_shim_batch_shares_fold_arrays_and_reports_per_job_status(shim_cpu, tmp_path):
    from conftest import write_problem_bin
    init, deg, ei, ej, ed, et = small_problem(50, 4, 0.2, 3)
    hold = (np.array([0, 3, 7], np.int32), np.array([5, 9, 11], np.int32), np.array([1.5, 2.5, 0.25]))
    write_problem_bin(tmp_path / "p.bin", init, deg, ei, ej, ed, et, hold)
    r = _harness(shim_cpu, "batch", tmp_path / "p.bin", tmp_path / "o.bin", 5, 250, 4.0, 0.01, 0.02, 1e-4, 5, 3, 1)
    _clean(r)
    assert r["n"] == 5 and r["names"][:8] == ["converged", "iterations", "final_mae", "final_k", "holdout_sum_abs",
                                               "holdout_count", "status", "message"]
    assert "shared=4" in r["jobs"][0]["message"]             # the four other jobs carried the same edge vectors
    assert [j["status"] for j in r["jobs"]] == [0] * 5 and all(j["pos_len"] == 200 for j in r["jobs"])
    out = np.fromfile(tmp_path / "o.bin").reshape(5, 7 + 200)
    for j in range(5):
        assert out[j, 1] == 247 and out[j, 3] == pytest.approx(4.0 * (1 + 0.25 * j) * 0.99 + 0.02 + 1e-4, rel=1e-15)
        assert out[j, 4] == pytest.approx(hold[2].sum() + hold[0].sum() + 2 * hold[1].sum()) and out[j, 5] == 3
    r = _harness(shim_cpu, "batch", tmp_path / "p.bin", tmp_path / "o.bin", 2, 250, 4.0, 0.01, 0.02, 1e-4, 5, 3, 0)
    assert all(j["pos_len"] == 0 for j in r["jobs"])         # positions stay on the device side unless asked for


# ------------------------------------------------------------------ parsing and the sparse entry --
def _odd_cells(m, seed):
    if seed % 2:
        m[3, 4] = m[4, 3] = "NA"; m[5, 6] = m[6, 5] = "abc"; m[7, 8] = m[8, 7] = ">"; m[1, 2] = "  3.5"; m[2, 1] = "3.5e0"
        m[9, 10] = np.nan; m[10, 9] = float("nan"); m[11, 12] = 4; m[12, 11] = np.float32(4); m[13, 14] = "<1e-3"; m[14, 13] = "> 2"
    return m


@pytest.mark.parametrize("seed", range(4))
def test_vectorised_parsing_equals_the_cell_by_cell_rule(seed):
    """R/core.R:345-374 (startsWith / sub / as.numeric) without a Python loop over the cells: same value, threshold
    code and NA mask as the cell-by-cell rule and as the R-glue restatement, for object and for string matrices."""
    m = _odd_cells(random_r_matrix(60, 0.3, seed), seed)
    got = core.parse_values(m)
    want = core._parse_elementwise(np.asarray(m).ravel())
    for a, b in zip(got, want):
        assert np.array_equal(a, b, equal_nan=True)
    ms = np.where(np.frompyfunc(lambda x: x is None, 1, 1)(m).astype(bool), "NA", m).astype(str)
    for a, b in zip(core.parse_values(ms), core._parse_elementwise(ms.ravel())):
        assert np.array_equal(a, b, equal_nan=True)
    value, code, is_na = core.parse_dissimilarity(m)
    rv, rc, rna = r_glue.parse_matrix(m)
    assert np.array_equal(is_na, rna) and np.array_equal(code[~rna], rc[~rna])
    assert np.array_equal(np.where(np.isnan(value) | is_na, np.inf, value), np.where(np.isnan(rv), np.inf, rv))


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("preserve", [True, False])
def test_sparse_table_builds_the_same_problem_as_the_matrix(seed, preserve):
    """build_problem_coo: degrees, order and the edge list (in which(arr.ind = TRUE) order) of the dense path,
    from the non-NA cells listed in any order, in both or in one orientation."""
    m = random_r_matrix(70, 0.25, seed)
    dense = core.build_problem(m, preserve)
    ii, jj = np.nonzero(np.frompyfunc(lambda x: x is not None, 1, 1)(m).astype(bool))
    off = ii != jj
    perm = np.random.default_rng(seed).permutation(int(off.sum()))
    ii, jj = ii[off][perm], jj[off][perm]
    for sel in (np.ones(len(ii), bool), ii < jj, ii > jj):
        coo = core.build_problem_coo(70, ii[sel], jj[sel], m[ii[sel], jj[sel]], preserve)
        for k in ("degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh"):
            assert np.array_equal(dense[k], coo[k]), k
        assert (dense["order"] is None) == (coo["order"] is None)
        assert dense["order"] is None or np.array_equal(dense["order"], coo["order"])
    with pytest.raises(ValueError, match="out of range"):
        core.build_problem_coo(70, [0, 70], [1, 2], [1.0, 2.0])


# ------------------------------------------------------------------ folds, subsampling -----------
def test_create_cv_folds_follows_the_reference_scheme():
    """cv.create_cv_folds vs the loop restatement of R/utils.R:103-147 fed the same draws; sizes, symmetry,
    disjoint folds, validation messages."""
    m = random_r_matrix(40, 0.4, 7)

    class Rec:                         # records what the product drew so that the restatement can replay it
        def __init__(self, seed): self.rng, self.picks = np.random.default_rng(seed), []
        def choice(self, a, size, replace): p = self.rng.choice(a, size=size, replace=replace); self.picks.append(p); return p

    rec = Rec(3)
    got = cv.create_cv_folds(m, n_folds=5, rng=rec)
    want, pool = r_glue.create_cv_folds(m, 5, rec.picks)
    assert len(got) == 5
    non_na = sum(x is not None for x in m.ravel())
    for f in range(5):
        assert len(rec.picks[f]) == non_na // 10
        g, w = got[f]["train"], want[f]
        assert all((a is None) == (b is None) and (a is None or a == b) for a, b in zip(g.ravel(), w.ravel()))
        na = np.frompyfunc(lambda x: x is None, 1, 1)(g).astype(bool)
        assert np.array_equal(na, na.T) and got[f]["truth"] is m
    held = [np.frompyfunc(lambda x: x is None, 1, 1)(got[f]["train"]).astype(bool) & ~np.frompyfunc(lambda x: x is None, 1, 1)(m).astype(bool) for f in range(5)]
    assert not np.any(sum(h.astype(int) for h in held) > 1)            # no cell is held out twice
    fm = np.where(np.frompyfunc(lambda x: x is None, 1, 1)(m).astype(bool), np.nan, 1.0)
    assert len(cv.create_cv_folds(fm, n_folds=4, random_seed=1)) == 4 and np.isnan(cv.create_cv_folds(fm, None, 4, 1)[0]["train"]).sum() > np.isnan(fm).sum()
    for kw, msg in ((dict(n_folds=1), "`n_folds` must be an integer greater than or equal to 2."),
                    (dict(n_folds=41), "`n_folds` cannot be larger than the number of rows in the matrix."),
                    (dict(random_seed=1.5), "`random_seed` must be an integer."),
                    (dict(ground_truth_matrix=np.zeros((3, 3))), "must have the same dimensions")):
        with pytest.raises(ValueError, match=re.escape(msg)):
            cv.create_cv_folds(m, **kw)


def test_folds_on_the_cell_list_equal_folds_on_the_matrix():
    """make_folds_cells / fold_problem_cells (nothing n x n) give the training problem, degrees and out-of-sample
    cells that masking the matrix gives (R/adaptive_sampling.R:2608-2647) for the same drawn cells."""
    n = 50
    m = random_r_matrix(n, 0.3, 2)
    value, code, is_na = core.parse_dissimilarity(m)
    ii, jj = np.nonzero(np.triu(~is_na, 1))
    full = core.build_problem_coo(n, ii, jj, m[ii, jj], preserve_order=True)
    folds = cv.make_folds_cells(n, full["cell_i"], full["cell_j"], 4, np.random.default_rng(0))
    assert [len(p) for p in folds] == [(n + 2 * len(ii)) // 8] * 4
    seen = np.zeros(n + 2 * len(ii), dtype=int)
    for picks in folds:
        seen[picks] += 1
        pr = picks[picks >= n] - n
        seen[n + (pr ^ 1)] += 1
        a = np.where(picks < n, picks, full["cell_i"][np.maximum(picks - n, 0) >> 1])
        b = np.where(picks < n, picks, full["cell_j"][np.maximum(picks - n, 0) >> 1])
        swap = (picks >= n) & (((picks - n) & 1) == 1)
        a, b = np.where(swap, b, a), np.where(swap, a, b)
        pm, hi_m, hj_m, ht_m = cv._fold_job(value, code, is_na, a + b * n, True)
        pc, hi_c, hj_c, ht_c = cv.fold_problem_cells(full, picks, n)
        for k in ("degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh"):
            assert np.array_equal(pm[k], pc[k]), k
        assert sorted(zip(hi_m.tolist(), hj_m.tolist(), ht_m.tolist())) == sorted(zip(hi_c.tolist(), hj_c.tolist(), ht_c.tolist()))
    assert seen.max() <= 2 and np.all(seen[:n] <= 1)              # a pair leaves the pool with its mirror (drawn + mirrored at most once each way)


def _scipy_components(n, ei, ej, masks):
    """Stand-in for _lib.components on a box without a GPU (tests of the HOST logic only)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    masks = np.ones((1, n), bool) if masks is None else np.asarray(masks, bool)
    comp, pts, edg = [], [], []
    for mk in masks:
        keep = mk[ei] & mk[ej]
        g = coo_matrix((np.ones(keep.sum()), (ei[keep], ej[keep])), shape=(n, n))
        lab = connected_components(g, directed=False)[1]
        comp.append(len(set(lab[mk]))); pts.append(int(mk.sum())); edg.append(int(keep.sum()))
    return np.array(comp), np.array(pts), np.array(edg)


def test_subsampling_follows_the_reference_loop():
    from topolow_b200 import subsample
    m = random_r_matrix(60, 0.13, 11, thresholds=False)               # sparse: some attempts are disconnected
    fm = np.where(np.frompyfunc(lambda x: x is None, 1, 1)(m).astype(bool), np.nan, 1.0) * np.array(
        [[0.0 if x is None else float(x) for x in row] for row in m])
    np.fill_diagonal(fm, 0.0)
    want_full = r_glue.check_matrix_connectivity(fm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got_full = subsample.check_matrix_connectivity(fm, components_fn=_scipy_components)
    assert got_full["n_components"] == want_full["n_components"] and got_full["is_connected"] == want_full["is_connected"]
    assert got_full["completeness"] == pytest.approx(want_full["completeness"]) and got_full["n_measurements"] == want_full["n_measurements"]
    hits = 0
    for seed in range(12):
        for preserve in (False, True):
            rng = np.random.default_rng(seed)
            attempts = [rng.choice(60, size=25, replace=False) for _ in range(5)]
            if preserve:
                attempts = [np.sort(a) for a in attempts]
            want = r_glue.subsample_dissimilarity_matrix(fm, attempts)
            try:
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    got = subsample.subsample_dissimilarity_matrix(fm, 25, rng=np.random.default_rng(seed), preserve_order=preserve,
                                                                   components_fn=_scipy_components)
            except RuntimeError as e:
                assert want is None and "Failed to obtain a connected subsample after 5 attempts." in str(e)
                continue
            hits += 1
            assert want is not None and got["attempt_number"] == want[0] and np.array_equal(got["selected_indices"], want[1])
            assert got["completeness"] == pytest.approx(want[2]["completeness"]) and got["is_connected"]
            assert np.array_equal(got["subsampled_matrix"], fm[np.ix_(want[1], want[1])], equal_nan=True)
    assert hits > 0
    whole = subsample.subsample_dissimilarity_matrix(fm, 60, components_fn=_scipy_components)
    assert whole["attempt_number"] == 1 and np.array_equal(whole["selected_indices"], np.arange(60))
    with pytest.raises(ValueError, match="sample_size must be a numeric value >= 2"):
        subsample.subsample_dissimilarity_matrix(fm, 1, components_fn=_scipy_components)
    chk = subsample.sanity_check_subsample(fm[:30, :30], folds=20, verbose=False)
    assert not chk["checks"]["sufficient_points"] and "Very few points (30) for 20-fold CV." in chk["warnings"][0]
    assert chk["diagnostics"]["n_measurements"] == int((~np.isnan(fm[:30, :30])).sum() / 2)


# ------------------------------------------------------------------ the sampler between fits ------
def _sample_table(rows, seed):
    rng = np.random.default_rng(seed)
    t = {"log_N": rng.uniform(0.7, 2.3, rows), "log_k0": rng.uniform(0, 3, rows), "log_cooling_rate": rng.uniform(-7, -3, rows),
         "log_c_repulsion": rng.uniform(-8, -2, rows)}
    t["Holdout_MAE"] = 0.8 + 0.3 * (t["log_N"] - 1.6) ** 2 + 0.1 * rng.random(rows)
    t["Holdout_MAE"][::17] = np.nan
    t["Holdout_MAE"][5] = 40.0                      # an outlier the MAD rule removes
    t["NLL"] = 100 * (1 + np.log(2 * t["Holdout_MAE"]))
    return t


def test_weighted_marginals_and_kde_draws_follow_the_reference():
    """sampler.weighted_kde / calculate_weighted_marginals / generate_kde_samples (one broadcast) vs the loop
    restatement of R/adaptive_sampling.R:1901-1935, :2457-2519, :1804-1885 with the same uniform draws."""
    from topolow_b200 import sampler
    t = _sample_table(90, 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = sampler.calculate_weighted_marginals(t)
    want = r_glue.calculate_weighted_marginals(t)
    for v in sampler.PAR_NAMES:
        np.testing.assert_allclose(got[v]["x"], want[v]["x"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(got[v]["y"], want[v]["y"], rtol=1e-10, atol=1e-300)
        assert len(got[v]["x"]) == 512
    # the weights favour low MAE: the log_N marginal peaks near the minimum of the MAE parabola
    assert abs(got["log_N"]["x"][np.argmax(got["log_N"]["y"])] - 1.6) < 0.35
    assert np.array_equal(np.isnan(sampler.clean_data(t["Holdout_MAE"])), np.isnan(np.array(r_glue.clean_data(list(t["Holdout_MAE"])))))

    class Rec:                                      # hands out recorded uniforms in the order the product asks for them
        def __init__(self): self.rng, self.u = np.random.default_rng(4), []
        def random(self, n=None):
            v = self.rng.random(n)
            if n is not None: self.u.append(v)
            return v
    rec = Rec()
    new = sampler.generate_kde_samples(t, 25, epsilon=0.3, rng=rec)
    ref = r_glue.generate_kde_samples(t, 25, dict(zip(sampler.PAR_NAMES, rec.u)))
    for v in sampler.PAR_NAMES:
        np.testing.assert_allclose(new[v], ref[v], rtol=1e-9)
        assert new[v].min() >= got[v]["x"][0] - 1e-9 and new[v].max() <= got[v]["x"][-1] + 1e-9
    with pytest.raises(ValueError, match="Missing required columns: log_k0"):
        sampler.calculate_weighted_marginals({k: v for k, v in t.items() if k != "log_k0"})
    with pytest.raises(ValueError, match="must contain a 'Holdout_MAE' column"):
        sampler.generate_kde_samples({"log_N": np.zeros(3)}, 2)


def test_lhs_design_and_batched_chains():
    from topolow_b200 import sampler
    d = sampler.lhs_design(40, (2, 10), (1.0, 20.0), (1e-4, 0.05), (1e-4, 0.05), rng=np.random.default_rng(0))
    assert d["N"].min() >= 2 and d["N"].max() <= 10 and d["N"].dtype.kind == "i"
    for k, (lo, hi) in (("k0", (1.0, 20.0)), ("c_repulsion", (1e-4, 0.05)), ("cooling_rate", (1e-4, 0.05))):
        strata = np.floor((d[k] - lo) / (hi - lo) * 40).astype(int)
        assert sorted(strata) == list(range(40))                     # one point per stratum: a Latin hypercube
    t = _sample_table(60, 2)
    calls = []

    def evaluate(matrix, sets):
        calls.append(len(sets))
        out = []
        for s in sets:
            mae = 0.8 + 0.3 * (math.log(s["N"]) - 1.6) ** 2
            out.append(dict(Holdout_MAE=mae if s["k0"] < 15 else math.nan, NLL=10.0, mean_iter=50.0, pct_converged=100.0))
        return out
    grown = sampler.adaptive_mc_batch(t, None, iterations=5, chains=8, mapping_max_iter=10, relative_epsilon=1e-4,
                                      rng=np.random.default_rng(3), evaluate=evaluate)
    assert calls == [8] * 5                                           # one batch per round, all chains in it
    added = len(grown["Holdout_MAE"]) - 60
    assert 0 < added <= 40 and all(len(v) == 60 + added for v in grown.values())
    assert np.all(np.exp(grown["log_N"][60:]).round() >= 1)
    with pytest.raises(ValueError, match="Samples file missing required columns: NLL"):
        sampler.adaptive_mc_batch({k: v for k, v in t.items() if k != "NLL"}, None, 1, 2, 10, 1e-4, evaluate=evaluate)


def test_series_weight_constant_is_shared_by_the_probe_and_the_tensor_pass():
    """rowblock_tc2.cuh computes the repulsion weight (d + 0.01)^-3 of a pair from S = d^2 / 2 with one rsqrt and a cubic
    (src/optimization.cpp:257-267 is the formula it stands for).  The constants are read from the source: for every
    pair the series form accepts (S >= kSeriesNearS, i.e. d >= 0.1) the result is within 1.2e-5 of the formula - far inside
    the TF32 rounding (4.9e-4) the weight gets next -, the probe in image_tc_kernel counts near pairs of the series form
    against the same constant, and the two-MUFU form's constants restate the same formula."""
    import re
    src = open(os.path.join(ROOT, "topolow_b200", "csrc", "rowblock_tc2.cuh")).read()
    m = re.search(r"float pl = fmaf\(([-0-9.e+]+)f, q, ([-0-9.e+]+)f\);\s*pl = fmaf\(pl, q, ([-0-9.e+]+)f\);\s*pl = fmaf\(pl, q, ([-0-9.e+]+)f\);", src)
    assert m, "series polynomial not found"
    c3, c2, c1, c0 = (float(x) for x in m.groups())
    consts = re.findall(r"constexpr float kSeriesNearS = ([0-9.e+-]+)f;", src)
    assert len(consts) == 1 and float(consts[0]) == 0.005
    s_min = float(consts[0])
    assert re.search(r"0\.5f \* d2 < fmaxf\(3\.01e-3f \* h_hi, kSeriesNearS\)", src), "the probe does not use kSeriesNearS"
    assert re.search(r"if \(series\) thr\[r\] = fmaxf\(thr\[r\], kSeriesNearS\);", src), "the pass does not use kSeriesNearS"
    d = np.concatenate([np.geomspace(np.sqrt(2 * s_min), 1e4, 20001), np.linspace(0.1, 0.3, 5001)])
    S = 0.5 * d * d
    q = 1.0 / np.sqrt(S)
    w = q ** 3 * (((c3 * q + c2) * q + c1) * q + c0)
    want = (d + 0.01) ** -3
    assert np.abs(w / want - 1).max() < 1.2e-5, np.abs(w / want - 1).max()
    m2 = re.search(r"rcp_approx_ftz\(fmaf\(sqrt_approx\(fabsf\([^;]*\)\)\), ([0-9.]+)f, ([0-9.]+)f\)\)", src)
    assert m2, "two-MUFU form not found"
    a, b = float(m2.group(1)), float(m2.group(2))
    assert np.abs((1.0 / (np.sqrt(S) * a + b)) ** 3 / want - 1).max() < 1e-7


def test_tensor_form_arithmetic_emulated_in_numpy():
    """The arithmetic of the two-GEMM repulsion pass (rowblock_tc2.cuh) restated in numpy, number format by number format,
    against the FP64 sums of src/optimization.cpp:257-281 seen from one endpoint: coordinates minus the centre split into
    a TF32 part (round to nearest) and a remainder (truncated by the tensor core), S = h_i + h_j - x_i . x_j from the
    three products hi x hi, hi x lo, lo x hi accumulated in FP32, near pairs (S < 3.01e-3 h_i or S < 0.005) from FP32
    differences, weights by rsqrt + cubic and truncated to TF32, sums of w x_j (x_j rounded to TF32) and of w, force =
    sum w x_j - x_i sum w.  Bars: every far pair's S within 2.5e-4 of d^2 / 2, every weight within 1.5e-3 of
    (d + 0.01)^-3, a row's repulsion sum within 1e-3 of the FP64 sum relative to its length (median 4e-4)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import tc2_arith_model as model
    rng = np.random.default_rng(11)
    n, d = 1200, 16
    centres = rng.normal(size=(4, d)) * 4
    X = (centres[rng.integers(0, 4, n)] + rng.normal(size=(n, d)) + np.linspace(0, 6, n)[:, None] * rng.normal(size=d) / 4).astype(np.float32)
    X = X + np.float32(30.0)             # far from the origin: the kernel works on coordinates minus the centre
    x, xp, _ = model.image(X)
    S, h_hi = model.distances(x, xp)
    x64 = X.astype(np.float64)
    diff = x64[None, :, :] - x64[:, None, :]                    # x_j - x_i
    d2 = (diff ** 2).sum(2)
    dist = np.sqrt(d2)
    off = ~np.eye(n, dtype=bool)
    near = model.near_mask(S, h_hi, series=True)
    far = off & ~near
    assert far.sum() > 0.99 * off.sum()                         # a spread-out map: near pairs are rare
    assert np.abs(S[far] / (0.5 * d2[far]) - 1).max() < 2.5e-4
    w = model.weights(S, series=True)
    want_w = (dist + 0.01) ** -3
    assert np.abs(w[far] / want_w[far] - 1).max() < 1.5e-3
    # near pairs: FP32 differences, exactly the FP32 form's arithmetic (in FP64 in the model: they are not what is being tested)
    force = model.tensor_pass(X, series=True)
    want = (np.where(off, want_w, 0.0)[:, :, None] * diff).sum(1)
    rel = np.linalg.norm(force - want, axis=1) / np.linalg.norm(want, axis=1)
    assert np.median(rel) < 4e-4 and rel.max() < 1e-3, (np.median(rel), rel.max())


def test_tc2_pipeline_protocol_model_under_random_interleavings():
    """The hand-off protocol of repulse_tc2_kernel (copy warp, MMA warp, eight consumer warps, bulk copies, the in-order
    tensor pipe, 18 mbarriers, the item ring) restated as a discrete-event model (tests/tc2_protocol_model.py) and run under
    random schedules over random item shapes - one-stage items, items shorter than the stage ring, CTAs that draw
    scattered item numbers: no deadlock, no barrier two phases ahead of a waiter, no buffer overwritten before its readers
    were done.  Without the rule that item 1 is published only after the GEMM 1s of item 0 the model finds the hang."""
    import random
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import tc2_protocol_model as model
    rng = random.Random(7)
    cases = []
    for seed in range(320):
        n_items = rng.randint(1, 10)
        shapes = [[rng.randint(1, 5) for _ in range(rng.randint(1, 3))] for _ in range(n_items)]
        if seed % 4 == 0:
            shapes = [[1] for _ in range(n_items)]
        if seed % 7 == 0:
            shapes = [[rng.randint(1, 2)] * rng.randint(1, 2) for _ in range(n_items)]
        cases.append((seed, shapes, rng.choice([0.0, 0.3, 0.7])))
    done = sum(model.run(seed, shapes, skip_prob=sp).stages_done for seed, shapes, sp in cases)
    assert done > 3000
    hangs = 0
    for seed, shapes, sp in cases:
        try:
            model.run(seed, shapes, skip_prob=sp, first_item_guard=False)
        except AssertionError as e:
            assert "ran ahead of a waiter" in str(e), e
            hangs += 1
    assert hangs > 0
