"""Row-block jobs in fit batches on the device: each is bit for bit the single row-block fit (`fit(mode=MODE_ROWBLOCK)`),
failures stay per job, the coloured jobs of a mixed batch are what the batch of those jobs alone returns, the device
list changes nothing, positions can stay on the library's side, an interrupt stops a running row-block job within a
few iterations and keeps queued ones from starting, and the .Call shim's 11th job element reaches the library."""
import json
import subprocess
import time

import numpy as np
import pytest

from conftest import small_problem
from topolow_b200 import _lib

pytestmark = pytest.mark.gpu

FIELDS = ("final_mae", "final_k", "iterations", "iterations_run", "converged", "pair_updates", "holdout_sum_abs",
          "holdout_count", "status")
RB = _lib.MODE_ROWBLOCK


def _holdout(n, seed, cells=60):
    rng = np.random.default_rng(seed)
    return rng.integers(0, n, cells).astype(np.int32), rng.integers(0, n, cells).astype(np.int32), rng.uniform(1, 6, cells)


def _job(a, n_iter, seed, hold=None, eps=1e-4, window=5, freq=3, **kw):
    return dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4], edge_thresh=a[5],
                n_iter=n_iter, k0=4.0 + 0.1 * seed, cooling_rate=0.01, c_repulsion=0.02, relative_epsilon=eps,
                convergence_window=window, convergence_check_freq=freq, seed=seed, holdout=hold, **kw)


def _single(job):
    """The same job as one topolow_fit call."""
    j = dict(job)
    args = [j.pop(k) for k in ("initial_positions", "degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh", "n_iter", "k0",
                               "cooling_rate", "c_repulsion", "relative_epsilon", "convergence_window",
                               "convergence_check_freq")]
    return _lib.fit(*args, **j)


def _same(x, y, positions=True):
    assert x["status"] == y["status"], (x.get("message"), y.get("message"))
    if x["status"] != _lib.OK and "final_mae" not in x:
        assert x == y
        return
    assert all(x[k] == y[k] for k in FIELDS), [(k, x[k], y[k]) for k in FIELDS if x[k] != y[k]]
    if positions:
        assert np.array_equal(x["positions"], y["positions"])
    if "trace_mae" in x and "trace_mae" in y:
        assert np.array_equal(x["trace_mae"], y["trace_mae"], equal_nan=True)


def sparse_problem(n, d, per_point, seed):
    """A large random map in edge-list form without an n x n intermediate: about per_point measured pairs per point."""
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, d)) * 3
    a, b = rng.integers(0, n, n * per_point), rng.integers(0, n, n * per_point)
    a, b = np.minimum(a, b), np.maximum(a, b)
    key = np.unique((a * n + b)[a != b])
    ei, ej = (key // n).astype(np.int32), (key % n).astype(np.int32)
    ed = np.maximum(np.linalg.norm(X[ei] - X[ej], axis=1) * (1 + 0.05 * rng.normal(size=len(ei))), 0.1)
    et = np.zeros(len(ei), np.int32)
    deg = (np.bincount(ei, minlength=n) + np.bincount(ej, minlength=n) + 1).astype(np.int32)
    init = np.vstack([np.zeros((1, d)), np.cumsum(rng.uniform(0, 2 * ed.max() / n, size=(n - 1, d)), axis=0)])
    return init, deg, ei, ej, ed, et


def rowblock_jobs():
    """Maps of every kind the row-block policy handles, with hold-out cells and traces."""
    p8 = small_problem(3000, 8, 0.01, 81)            # the policy moves from the FP32 start to the tensor form
    p3 = small_problem(800, 3, 0.05, 31)             # thresholds (small_problem draws them), FP32 form
    p20 = small_problem(1500, 20, 0.03, 201)         # difference form, ndim 17..32
    p32 = small_problem(700, 32, 0.05, 321)
    return [
        _job(p8, 80, 1, _holdout(3000, 1), mode=RB, trace=True),
        _job(p3, 120, 2, _holdout(800, 2), mode=RB, trace=True),
        _job(p20, 60, 3, _holdout(1500, 3), mode=RB, trace=True),
        _job(p32, 60, 4, _holdout(700, 4), mode=RB, trace=True),
        _job(p3, 300, 5, _holdout(800, 5), eps=0.5, window=2, mode=RB, trace=True),        # converges early
        _job(p8, 90, 6, _holdout(3000, 6), window=91, mode=RB, trace=True),                # runs all its iterations
    ]


def coloured_jobs(count, n_iter=40):
    probs = [small_problem(n, d, 0.1, 7 + d) for n, d in ((220, 2), (300, 3), (260, 5))]
    return [_job(probs[j % 3], n_iter, 100 + j, _holdout(len(probs[j % 3][1]), j) if j % 2 else None,
                 precision=_lib.PREC_F64_EXACT if j % 4 == 3 else _lib.PREC_F32) for j in range(count)]


def small_rowblock_jobs():
    a, b = small_problem(1200, 6, 0.03, 61), small_problem(900, 24, 0.04, 241)
    return [_job(a, 50, 11, _holdout(1200, 11), mode=RB), _job(b, 40, 12, _holdout(900, 12), mode=RB)]


def _too_few():
    return dict(initial_positions=np.zeros((1, 2)), degrees=np.ones(1, np.int32), edge_i=np.zeros(0, np.int32),
                edge_j=np.zeros(0, np.int32), edge_dist=np.zeros(0), edge_thresh=np.zeros(0, np.int32), n_iter=10, k0=4.0,
                cooling_rate=0.01, c_repulsion=0.02, mode=RB)


def test_rowblock_jobs_are_bit_for_bit_single_fits():
    jobs = rowblock_jobs()
    got = _lib.fit_batch(jobs)
    want = [_single(j) for j in jobs]
    for g, w in zip(got, want):
        assert g["status"] == _lib.OK
        _same(g, w)
        assert g["holdout_count"] > 0
    # again: the best state of a fit that stopped early must not depend on how many iterations the host had enqueued
    for g, w, g0 in zip(_lib.fit_batch(jobs), [_single(j) for j in jobs], got):
        _same(g, g0)
        _same(w, g0)
    assert want[4]["converged"] and want[4]["iterations_run"] < 300
    assert want[5]["iterations_run"] == 90 and not want[5]["converged"]


def test_failures_stay_per_job():
    ok_c = coloured_jobs(1)[0]
    ok_r = small_rowblock_jobs()[0]
    wide = _job(small_problem(300, 33, 0.1, 33), 10, 7, mode=RB)
    replay = _job(small_problem(100, 2, 0.2, 2), 10, 8, mode=_lib.MODE_REPLAY)
    a = list(small_problem(400, 4, 0.05, 44))
    a[2] = a[2].copy()
    a[2][5] = 400                                   # an edge that names a point the map does not have
    bad_edge = _job(a, 10, 9, mode=RB)
    jobs = [ok_c, _too_few(), wide, replay, bad_edge, ok_r]
    got = _lib.fit_batch(jobs)
    assert got[1]["status"] == _lib.ERR_TOO_FEW_POINTS
    for j in (2, 4):                                # the single fit's status and message
        with pytest.raises(_lib.TopolowError) as e:
            _single(jobs[j])
        assert got[j] == dict(status=e.value.status, message=str(e.value)), (got[j], e.value)
        assert got[j]["status"] == _lib.ERR_BAD_ARG
    assert "ndim <= 32" in got[2]["message"]
    assert got[3]["status"] == _lib.ERR_BAD_ARG and "coloured and row-block" in got[3]["message"]
    _same(got[0], _lib.fit_batch([ok_c])[0])
    _same(got[5], _single(ok_r))


@pytest.mark.parametrize("count", [20, 15])
def test_mixed_batches_keep_the_coloured_results(count):
    col = coloured_jobs(count)
    rb = small_rowblock_jobs()
    alone = _lib.fit_batch(col)
    mixed = _lib.fit_batch(rb[:1] + col + rb[1:])
    for x, y in zip(mixed[1:-1], alone):
        _same(x, y)
    for x, j in zip((mixed[0], mixed[-1]), rb):
        _same(x, _single(j))


def test_device_lists_change_nothing():
    jobs = small_rowblock_jobs()[:1] + coloured_jobs(17) + small_rowblock_jobs()[1:]
    want = _lib.fit_batch(jobs, device=0)
    for dev in ([0, 0], [0, 0, 0]):
        for x, y in zip(_lib.fit_batch(jobs, device=dev), want):
            _same(x, y)


def test_device_lists_change_nothing_for_a_rowblock_grid():
    # 64 ndim-24 fold fits of one 5 000-point map: four shares on one device returned other best positions for a few
    # jobs while their row-block fits ran side by side
    from tools import synth
    prob = synth.make_problem(5000, 24, 0.95, seed=1)
    ei, ej, ed, et = prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"]
    which = np.random.default_rng(5).integers(0, 8, len(ei))
    jobs = []
    for f in range(4):
        held = (which == f) & (et == 0)
        tr = ~held
        deg = (np.bincount(ei[tr], minlength=5000) + np.bincount(ej[tr], minlength=5000) + 1).astype(np.int32)
        a = (prob["initial_positions"], deg, ei[tr], ej[tr], ed[tr], et[tr])
        jobs += [_job(a, 250, 16 * f + s, (ei[held], ej[held], ed[held]), mode=RB) for s in range(16)]
    want = _lib.fit_batch(jobs)
    for dev in ([0, 0], [0, 0, 0, 0]):
        for x, y in zip(_lib.fit_batch(jobs, device=dev), want):
            _same(x, y)


def test_null_positions_give_the_same_sums():
    jobs = small_rowblock_jobs() + coloured_jobs(3)
    want = _lib.fit_batch(jobs)
    got = _lib.fit_batch(jobs, keep_positions=False)
    for x, y in zip(got, want):
        assert "positions" not in x
        _same(x, y, positions=False)
        assert x["holdout_count"] > 0 or y["holdout_count"] == 0


def _interrupted(jobs, **kw):
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, **kw)
    assert e.value.status == _lib.ERR_INTERRUPTED and len(e.value.results) == len(jobs)
    return e.value.results


@pytest.mark.parametrize("at", [1, 2, 3, 4])
def test_interrupt_before_and_after_set_up(at):
    # polls 1 and 2: before and after the batch's set-up; 3 and 4: before and after the first row-block job's set-up
    # (a batch of row-block jobs only has no coloured launch to wait on in between)
    jobs = small_rowblock_jobs() + [_too_few()] + (coloured_jobs(2) if at <= 2 else [])
    calls = []
    res = _interrupted(jobs, interrupt=lambda: (calls.append(1), len(calls) >= at)[1])
    assert len(calls) == at
    for job, r in zip(jobs, res):
        if len(job["degrees"]) < 2:
            assert r["status"] == _lib.ERR_TOO_FEW_POINTS
            continue
        assert r["status"] == _lib.ERR_INTERRUPTED and r["message"] == "interrupted"
        assert r["iterations_run"] == 0 and r["pair_updates"] == 0
        if job.get("mode") == RB:
            assert np.array_equal(r["positions"], job["initial_positions"])
        else:
            np.testing.assert_allclose(r["positions"], job["initial_positions"], rtol=1e-6, atol=1e-6)   # FP32 image


def test_interrupt_while_coloured_fits_run_before_a_rowblock_job():
    # the row-block job is set up once the coloured fits have ended; until then the batch keeps polling, so an interrupt
    # one period after set-up stops the coloured fits and the row-block job does not start
    a = small_problem(3000, 3, 0.01, 31)
    col = [_job(a, 3000, j, _holdout(3000, j), window=3001) for j in range(3)]
    rb = small_rowblock_jobs()[0]
    calls = []

    def poll():
        calls.append(time.perf_counter())
        return len(calls) > 2 and calls[-1] - calls[1] > 0.1     # 0.1 s after the poll that follows the set-up

    t0 = time.perf_counter()
    res = _interrupted(col + [rb], interrupt=poll)
    wall = time.perf_counter() - t0
    for j, r in zip(col, res[:3]):
        assert r["status"] == _lib.ERR_INTERRUPTED and 0 < r["iterations_run"] < j["n_iter"], r["iterations_run"]
    assert res[3]["status"] == _lib.ERR_INTERRUPTED and res[3]["iterations_run"] == 0
    assert wall < 1.5, wall
    assert max(np.diff(calls[1:])) < 0.1             # polled at least every 100 ms after the set-up


def test_a_running_rowblock_job_stops_within_ten_iterations():
    # ndim 20: the difference form in every iteration, so iterations cost the same from the first to the last
    big = sparse_problem(20000, 20, 8, 9)
    job = _job(big, 3000, 31, window=3001, mode=RB)
    full = _single(job)
    tau = full["device_ms"] * 1e-3 / full["iterations_run"]     # seconds per iteration, launched back to back
    calls = []

    def poll():                                       # polls 1..4: before and after the batch's and the job's set-up
        calls.append(time.perf_counter())
        return len(calls) > 4 and calls[-1] - calls[3] > 0.3

    r = _interrupted([job], interrupt=poll)[0]
    done_at_fire = (calls[-1] - calls[3]) / tau      # an upper bound of the iterations completed when the poll fired
    assert r["status"] == _lib.ERR_INTERRUPTED
    assert 1 <= r["iterations_run"] <= done_at_fire + 10 + 2, (r["iterations_run"], done_at_fire)


def _after(seconds):
    t0 = time.perf_counter()
    return lambda: time.perf_counter() - t0 > seconds


def test_interrupt_while_a_rowblock_job_runs():
    big = sparse_problem(20000, 16, 8, 7)
    n_iter = 12000
    run = _job(big, n_iter, 21, _holdout(20000, 21), window=n_iter + 1, mode=RB, trace=True)   # cannot stop early
    queued = _job(big, 50, 22, mode=RB)
    short = coloured_jobs(1, n_iter=20)[0]
    t0 = time.perf_counter()
    full = _single(run)
    t_full = time.perf_counter() - t0
    assert t_full > 2.0, t_full
    got = _interrupted([short, run, queued], interrupt=_after(0.5))
    _same(got[0], _lib.fit_batch([short])[0])     # had ended: bit for bit
    r = got[1]
    assert r["status"] == _lib.ERR_INTERRUPTED and r["message"] == "interrupted"
    k = r["iterations_run"]
    assert 1 <= k < n_iter // 2, k
    assert r["pair_updates"] == k * 20000 * 19999 // 2
    assert np.array_equal(r["trace_mae"][:k], full["trace_mae"][:k], equal_nan=True)
    assert np.all(np.isnan(r["trace_mae"][k:]))
    assert np.all(np.isfinite(r["positions"]))
    q = got[2]
    assert q["status"] == _lib.ERR_INTERRUPTED and q["iterations_run"] == 0
    assert np.array_equal(q["positions"], queued["initial_positions"])


def test_interrupted_batches_release_everything():
    import torch
    jobs = coloured_jobs(3, n_iter=2000) + small_rowblock_jobs()
    for j in jobs:
        j["convergence_window"] = j["n_iter"] + 1
    jobs[-1]["n_iter"] = jobs[-1]["convergence_window"] = 3000
    before = _lib.fit_batch(jobs)
    free0 = None
    for rep in range(6):
        calls = []
        res = _interrupted(jobs, interrupt=lambda: (calls.append(1), len(calls) > 4)[1])   # fifth poll: fits running
        assert any(r["status"] == _lib.ERR_INTERRUPTED for r in res)
        torch.cuda.synchronize()
        if rep == 0:
            free0 = torch.cuda.mem_get_info()[0]
    assert torch.cuda.mem_get_info()[0] >= free0 - (8 << 20)
    for x, y in zip(_lib.fit_batch(jobs), before):      # nothing carried over
        _same(x, y)


# ---- the .Call shim with the real library ----
@pytest.fixture(scope="module")
def shim_gpu(tmp_path_factory):
    from conftest import build_r_shim_harness
    return build_r_shim_harness(str(tmp_path_factory.mktemp("shim") / "harness_gpu"), real_library=True)


def _run(exe, *args):
    out = subprocess.run([exe] + [str(x) for x in args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_r_shim_modes_and_keep_false_against_the_real_library(shim_gpu, tmp_path):
    from conftest import write_problem_bin
    init, deg, ei, ej, ed, et = small_problem(600, 5, 0.05, 23)
    held = np.random.default_rng(1).random(len(ei)) < 0.1
    hold = (ei[held], ej[held], ed[held])
    write_problem_bin(tmp_path / "p.bin", init, deg, ei[~held], ej[~held], ed[~held], et[~held], hold)
    hp = (60, 4.0, 0.01, 0.02, 1e-4, 5, 3)         # n_iter k0 cooling c_rep rel_eps window freq
    modes = ("rowblock", "-", "coloured", "rowblock")
    res = {}
    for keep in (1, 0):
        r = _run(shim_gpu, "batch_modes", tmp_path / "p.bin", tmp_path / f"k{keep}.bin", len(modes), *hp, keep, *modes)
        assert r["left_by"] == "return" and r["protect_depth"] == 0 and r["errors"] == 0
        assert [j["status"] for j in r["jobs"]] == [0] * len(modes)
        res[keep] = np.fromfile(tmp_path / f"k{keep}.bin")
    n, d = init.shape
    with_pos = res[1].reshape(len(modes), 7 + n * d)
    sums = res[0].reshape(len(modes), 7)
    assert np.array_equal(with_pos[:, :7], sums)     # MAE, iterations, hold-out sums: the same without positions
    assert np.all(sums[:, 5] > 0)
    # the ctypes path with the shim's seeds (the stand-in runtime's RNG draws 0.25, 0.5) and parameters
    seed0 = ((1 << 30) << 32) | (1 << 31)
    jobs = []
    for j, m in enumerate(modes):
        jobs.append(dict(initial_positions=init, degrees=deg, edge_i=ei[~held], edge_j=ej[~held], edge_dist=ed[~held],
                         edge_thresh=et[~held], n_iter=hp[0], k0=hp[1] * (1.0 + 0.25 * j), cooling_rate=hp[2],
                         c_repulsion=hp[3], relative_epsilon=hp[4], convergence_window=hp[5], convergence_check_freq=hp[6],
                         seed=seed0 + j, holdout=hold, mode=RB if m == "rowblock" else _lib.MODE_COLOURED))
    for row, r in zip(with_pos, _lib.fit_batch(jobs)):
        want = [float(r["converged"]), r["iterations"], r["final_mae"], r["final_k"], r["holdout_sum_abs"],
                r["holdout_count"], r["status"]]
        assert np.array_equal(row[:7], np.array(want, dtype=np.float64))
        assert np.array_equal(row[7:].reshape(d, n).T, r["positions"])
