"""topolow_fit_batch_devices on the device: whatever the device list, every job's result is bit for bit what the plain
batch returns on the first device of the list; the one-CTA rule follows the job count of the whole call; the poll is
called from the calling thread only and an interrupt stops every share; bad lists are refused; nothing is left behind;
the .Call shim with a vector `device` returns what it returns with one ordinal."""
import threading

import numpy as np
import pytest
import torch

from conftest import small_problem
from test_gpu_batch_interrupt import _after, _holdout, _job, _same, mixed_jobs, multi_jobs
from topolow_b200 import _lib

pytestmark = pytest.mark.gpu

ONE_GPU_LISTS = ([0], [0, 0], [0, 0, 0])


def _free(device=0):
    torch.cuda.synchronize(device)
    return torch.cuda.mem_get_info(device)[0]


def _interrupted(jobs, **kw):
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, **kw)
    assert e.value.status == _lib.ERR_INTERRUPTED
    assert len(e.value.results) == len(jobs)
    return e.value.results


def test_every_device_list_gives_the_plain_batch():
    for jobs in (mixed_jobs(), multi_jobs(60)):
        want = _lib.fit_batch(jobs)
        for devices in ONE_GPU_LISTS:
            got = _lib.fit_batch(jobs, device=devices)
            assert len(got) == len(jobs)
            for x, y in zip(got, want):
                _same(x, y)
    mixed = _lib.fit_batch(mixed_jobs(), device=[0, 0])
    assert mixed[-1]["status"] == _lib.ERR_TOO_FEW_POINTS
    assert all(r["status"] == _lib.OK for r in mixed[:-1])


def test_split_batch_still_runs_every_fit_on_one_cta():
    # 19 jobs over three shares: no share reaches 16 jobs, but the call has 19, so every fit runs as a batch of 16 or
    # more runs it: one CTA with 64-point tiles (asked for explicitly here, on one device)
    jobs = mixed_jobs()
    one_cta = _lib.fit_batch([dict(j, max_ctas=1, tile_points=64) for j in jobs])
    got = _lib.fit_batch(jobs, device=[0, 0, 0])
    for x, y in zip(got, one_cta):
        _same(x, y)


def test_poll_is_called_from_the_calling_thread_only():
    jobs = mixed_jobs()
    want = _lib.fit_batch(jobs)
    threads = []
    got = _lib.fit_batch(jobs, device=[0, 0], interrupt=lambda: threads.append(threading.get_ident()) and False)
    assert len(threads) >= 2                               # before set-up and after it at least
    assert set(threads) == {threading.get_ident()}
    for x, y in zip(got, want):
        _same(x, y)


def test_interrupt_at_once_stops_every_share():
    for jobs in (mixed_jobs(), multi_jobs(60)):
        calls = []
        res = _interrupted(jobs, device=[0, 0], interrupt=lambda: (calls.append(1), True)[1])
        assert len(calls) == 1
        for job, r in zip(jobs, res):
            if len(job["degrees"]) < 2:
                assert r["status"] == _lib.ERR_TOO_FEW_POINTS
                continue
            assert r["status"] == _lib.ERR_INTERRUPTED and r["iterations_run"] == 0 and r["pair_updates"] == 0


def test_interrupt_after_set_up_stops_every_share_before_any_launch():
    jobs = mixed_jobs()
    calls = []
    res = _interrupted(jobs, device=[0, 0, 0], interrupt=lambda: (calls.append(1), len(calls) >= 2)[1])
    assert len(calls) == 2
    for job, r in zip(jobs, res):
        if len(job["degrees"]) >= 2:
            assert r["status"] == _lib.ERR_INTERRUPTED and r["iterations_run"] == 0
            np.testing.assert_allclose(r["positions"], job["initial_positions"], rtol=1e-6, atol=1e-6)


def _long_jobs():
    a, b = small_problem(3000, 3, 0.01, 31), small_problem(1200, 2, 0.02, 32)
    jobs = []
    for j in range(18):
        if j % 3 == 0:
            jobs.append(_job(a, 20, j, _holdout(a, j), window=21))
        elif j % 3 == 1:
            jobs.append(_job(a, 3000, j, _holdout(a, j), window=3001))
        else:
            jobs.append(_job(b, 1000, j, window=1001, precision=_lib.PREC_F64_EXACT))
    return jobs


def test_interrupt_while_the_fits_run_on_every_share():
    jobs = _long_jobs()
    want = _lib.fit_batch(jobs)
    _lib.fit_batch(jobs, device=[0, 0])                    # the pools of both shares are grown
    free0 = _free()
    got = _interrupted(jobs, device=[0, 0], interrupt=_after(0.5))
    assert _free() >= free0 - (8 << 20)
    assert all(r["status"] == _lib.OK for r in got[::3])
    stopped = [(j, r) for j, r in zip(jobs, got) if r["status"] == _lib.ERR_INTERRUPTED]
    assert stopped and any(r["iterations_run"] < j["n_iter"] / 2 for j, r in stopped)
    for j, r, w in zip(jobs, got, want):
        if r["status"] == _lib.OK:
            _same(r, w)
        else:
            assert r["status"] == _lib.ERR_INTERRUPTED and r["message"] == "interrupted"
            assert r["iterations_run"] < j["n_iter"]
            n = len(j["degrees"])
            assert r["pair_updates"] == r["iterations_run"] * n * (n - 1) // 2
            assert np.all(np.isfinite(r["positions"]))

    # several CTAs per fit: each fit stops where its CTA 0 runs the controller
    jobs = multi_jobs(4000, window=4001, freq=7)
    got = _interrupted(jobs, device=[0, 0], interrupt=_after(0.5))
    assert any(r["status"] == _lib.ERR_INTERRUPTED for r in got)
    for r in got:
        if r["status"] == _lib.ERR_INTERRUPTED:
            assert 0 < r["iterations_run"] < 4000
            assert r["iterations_run"] % 7 == 0 or r["iterations_run"] % 10 == 0, r["iterations_run"]


def test_interrupted_multi_device_batches_release_everything():
    jobs = mixed_jobs(3000, window=3001)
    before = _lib.fit_batch(jobs)
    free0 = None
    for rep in range(10):
        calls = []
        res = _interrupted(jobs, device=[0, 0], interrupt=lambda: (calls.append(1), len(calls) > 2)[1])
        assert len(calls) == 3 and any(r["status"] == _lib.ERR_INTERRUPTED for r in res)
        if rep == 0:
            free0 = _free()
    assert _free() >= free0 - (8 << 20)
    for x, y in zip(_lib.fit_batch(jobs, device=[0, 0]), before):      # no stale abort word, no state carried over
        _same(x, y)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("devices", [[0, 1], [1, 0, 1]])
def test_two_gpus_give_the_plain_batch_on_the_first(devices):
    for jobs in (mixed_jobs(), multi_jobs(60)):
        want = _lib.fit_batch(jobs, device=devices[0])
        _lib.fit_batch(jobs, device=devices)
        free0 = [_free(d) for d in (0, 1)]
        got = _lib.fit_batch(jobs, device=devices)
        for x, y in zip(got, want):
            _same(x, y)
        assert all(_free(d) >= f - (8 << 20) for d, f in zip((0, 1), free0))


@pytest.mark.parametrize("bad", [[], [-1], "count", [0, "count"]])
def test_bad_device_lists_are_refused(bad):
    count = torch.cuda.device_count()
    devices = [count if d == "count" else d for d in (bad if isinstance(bad, list) else [bad])]
    jobs = mixed_jobs()[:3]
    free0 = _free()
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, device=devices)
    assert e.value.status == _lib.ERR_BAD_ARG and "device" in str(e.value)
    assert _free() >= free0 - (1 << 20)


def test_r_shim_device_vector_against_the_real_library(tmp_path):
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
    a = run("batch_devices", tmp_path / "p.bin", tmp_path / "a.bin", *hp, "int", 0)
    b = run("batch_devices", tmp_path / "p.bin", tmp_path / "b.bin", *hp, "int", 0, 0)
    assert b["left_by"] == "return" and b["protect_depth"] == 0 and b["errors"] == 0 and b["interrupt_checks"] >= 2
    for k in ("interrupt_checks",):      # how often the library polled depends on timing
        a.pop(k), b.pop(k)
    assert a == b and [j["status"] for j in b["jobs"]] == [0, 0, 0]
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "b.bin").read_bytes()
