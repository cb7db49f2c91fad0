"""topolow_fit_batch_interruptible on the device: without an interrupt the batch is bit for bit the plain batch; an
interrupt before set-up, before the first launch or while the fits run stops the batch, reports finished jobs as
they are, stopped ones with status ERR_INTERRUPTED, and leaves nothing behind; the .Call shim leaves through
Rf_onintr."""
import time

import numpy as np
import pytest

from conftest import small_problem
from topolow_b200 import _lib

pytestmark = pytest.mark.gpu

FIELDS = ("final_mae", "final_k", "iterations", "iterations_run", "converged", "pair_updates", "holdout_sum_abs",
          "holdout_count", "status")


def _job(a, n_iter, seed, hold=None, window=5, freq=3, **kw):
    return dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4], edge_thresh=a[5],
                n_iter=n_iter, k0=4.0 + 0.1 * seed, cooling_rate=0.01, c_repulsion=0.02, relative_epsilon=1e-4,
                convergence_window=window, convergence_check_freq=freq, seed=seed, holdout=hold, **kw)


def _holdout(a, seed):
    rng = np.random.default_rng(seed)
    n = len(a[1])
    return rng.integers(0, n, 40).astype(np.int32), rng.integers(0, n, 40).astype(np.int32), rng.uniform(1, 6, 40)


def _too_few():
    return dict(initial_positions=np.zeros((1, 2)), degrees=np.ones(1, np.int32), edge_i=np.zeros(0, np.int32),
                edge_j=np.zeros(0, np.int32), edge_dist=np.zeros(0), edge_thresh=np.zeros(0, np.int32), n_iter=10, k0=4.0,
                cooling_rate=0.01, c_repulsion=0.02)


def mixed_jobs(n_iter=40, window=5):
    """18 one-CTA fits (grouped launches): FP32 and FP64, ndim 2, 3, 5, hold-out cells on every other job; plus a job
    with one point."""
    probs = [small_problem(n, d, 0.1, 7 + d) for n, d in ((220, 2), (300, 3), (260, 5))]
    jobs = []
    for j in range(18):
        a = probs[j % 3]
        prec = _lib.PREC_F64_EXACT if j % 4 == 3 else _lib.PREC_F32
        jobs.append(_job(a, n_iter, j, _holdout(a, j) if j % 2 else None, window=window, precision=prec))
    return jobs + [_too_few()]


def multi_jobs(n_iter, window=5, freq=3):
    """Two fits large enough to run on several CTAs each (a batch of fewer than 16 jobs)."""
    a = small_problem(6000, 4, 0.004, 5)
    return [_job(a, n_iter, s, _holdout(a, s) if s else None, window=window, freq=freq) for s in range(2)]


def _same(x, y):
    assert x["status"] == y["status"]
    if "positions" not in x:
        assert x == y
        return
    assert all(x[k] == y[k] for k in FIELDS), [(k, x[k], y[k]) for k in FIELDS if x[k] != y[k]]
    assert np.array_equal(x["positions"], y["positions"])


def _interrupted(jobs, **kw):
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, **kw)
    assert e.value.status == _lib.ERR_INTERRUPTED
    assert len(e.value.results) == len(jobs)
    return e.value.results


def test_never_firing_interrupt_is_bit_identical():
    for jobs in (mixed_jobs(), multi_jobs(60)):
        want = _lib.fit_batch(jobs)
        calls = []
        got = _lib.fit_batch(jobs, interrupt=lambda: calls.append(1) and False)
        assert len(calls) >= 2                       # before and after set-up at least
        for x, y in zip(got, want):
            _same(x, y)
    assert want[0]["status"] == _lib.OK and want[1]["status"] == _lib.OK


@pytest.mark.parametrize("at", [1, 2])
def test_interrupt_before_the_first_launch(at):
    for jobs in (mixed_jobs(), multi_jobs(60)):
        calls = []
        res = _interrupted(jobs, interrupt=lambda: (calls.append(1), len(calls) >= at)[1])
        assert len(calls) == at
        for job, r in zip(jobs, res):
            if len(job["degrees"]) < 2:
                assert r["status"] == _lib.ERR_TOO_FEW_POINTS
                continue
            assert r["status"] == _lib.ERR_INTERRUPTED and r["message"] == "interrupted"
            assert r["iterations_run"] == 0 and r["pair_updates"] == 0
            np.testing.assert_allclose(r["positions"], job["initial_positions"], rtol=1e-6, atol=1e-6)   # FP32 image


def _after(seconds):
    t0 = time.perf_counter()
    return lambda: time.perf_counter() - t0 > seconds


def test_interrupt_while_the_fits_run():
    # fits that cannot stop early (convergence_counter > mapping_max_iter, as the bench runs them); one in three is short
    # and ends long before the interrupt, the others would run for seconds
    a, b = small_problem(3000, 3, 0.01, 31), small_problem(1200, 2, 0.02, 32)
    jobs = []
    for j in range(18):
        if j % 3 == 0:
            jobs.append(_job(a, 20, j, _holdout(a, j), window=21))
        elif j % 3 == 1:
            jobs.append(_job(a, 3000, j, _holdout(a, j), window=3001))
        else:
            jobs.append(_job(b, 1000, j, window=1001, precision=_lib.PREC_F64_EXACT))
    t0 = time.perf_counter()
    want = _lib.fit_batch(jobs)
    t_full = time.perf_counter() - t0
    assert t_full > 2.0, t_full
    got = _interrupted(jobs, interrupt=_after(0.5))
    assert all(r["status"] == _lib.OK for r in got[::3])
    stopped = [(j, r) for j, r in zip(jobs, got) if r["status"] == _lib.ERR_INTERRUPTED]
    assert any(r["iterations_run"] < j["n_iter"] / 2 for j, r in stopped)
    for j, r, w in zip(jobs, got, want):
        if r["status"] == _lib.OK:
            _same(r, w)
        else:
            assert r["status"] == _lib.ERR_INTERRUPTED and r["iterations_run"] < j["n_iter"]
            n = len(j["degrees"])
            assert r["pair_updates"] == r["iterations_run"] * n * (n - 1) // 2    # as of the last completed iteration
            assert np.all(np.isfinite(r["positions"]))

    # several CTAs per fit: a fit stops where CTA 0 runs the controller
    jobs = multi_jobs(4000, window=4001, freq=7)
    got = _interrupted(jobs, interrupt=_after(0.5))
    assert any(r["status"] == _lib.ERR_INTERRUPTED for r in got)
    for r in got:
        if r["status"] == _lib.ERR_INTERRUPTED:
            assert 0 < r["iterations_run"] < 4000
            assert r["iterations_run"] % 7 == 0 or r["iterations_run"] % 10 == 0, r["iterations_run"]
    if any(r["status"] == _lib.OK for r in got):
        for r, w in zip(got, _lib.fit_batch(jobs)):
            if r["status"] == _lib.OK:
                _same(r, w)


def test_interrupted_batches_release_everything():
    import torch
    jobs = mixed_jobs(3000, window=3001)
    before = _lib.fit_batch(jobs)
    free0 = None
    for rep in range(20):
        calls = []
        res = _interrupted(jobs, interrupt=lambda: (calls.append(1), len(calls) > 2)[1])     # third poll: fits running
        assert len(calls) == 3 and any(r["status"] == _lib.ERR_INTERRUPTED for r in res)
        torch.cuda.synchronize()
        if rep == 0:
            free0 = torch.cuda.mem_get_info()[0]
    assert torch.cuda.mem_get_info()[0] >= free0 - (8 << 20)
    for x, y in zip(_lib.fit_batch(jobs), before):      # no stale abort word, no state carried over
        _same(x, y)


def test_r_shim_batch_interrupt_against_the_real_library(tmp_path):
    import json
    import subprocess
    from conftest import build_r_shim_harness, write_problem_bin
    exe = build_r_shim_harness(str(tmp_path / "harness_gpu"), real_library=True)
    init, deg, ei, ej, ed, et = small_problem(300, 3, 0.1, 21)
    held = np.random.default_rng(1).random(len(ei)) < 0.1
    write_problem_bin(tmp_path / "p.bin", init, deg, ei[~held], ej[~held], ed[~held], et[~held], (ei[held], ej[held], ed[held]))

    def run(*args):
        out = subprocess.run([exe] + [str(x) for x in args], capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr
        return json.loads(out.stdout.strip().splitlines()[-1])

    hp = (3, 40, 4.0, 0.01, 0.02, 1e-4, 5, 3, 1)
    r = run("batch_interrupt", tmp_path / "p.bin", tmp_path / "i.bin", *hp, 1)
    assert r["left_by"] == "Rf_onintr" and r["onintr_calls"] == 1 and r["interrupt_checks"] == 1
    assert r["raw_interrupt_jumps"] == 0 and r["protect_depth"] == 0 and r["errors"] == 0
    a = run("batch", tmp_path / "p.bin", tmp_path / "a.bin", *hp)
    b = run("batch_interrupt", tmp_path / "p.bin", tmp_path / "b.bin", *hp, 0)
    assert b["left_by"] == "return" and b["interrupt_checks"] >= 2 and b["onintr_calls"] == 0
    for k in ("scenario", "interrupt_checks"):      # how often the library polled depends on timing
        a.pop(k), b.pop(k)
    assert a == b and [j["status"] for j in b["jobs"]] == [0, 0, 0]
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "b.bin").read_bytes()
