"""CPU tests of row-block jobs in fit batches: the optional 11th job element of the .Call shim (integration/r_shim.c)
against the recording fake of the library (integration/r_stub/fake_topolow.c), and the `mode` plumbing of cv and
sampler down to every job of the batch."""
import json
import subprocess

import numpy as np
import pytest

from conftest import random_r_matrix, small_problem
from topolow_b200 import _lib, cv, sampler

BATCH_ARGS = (250, 4.0, 0.01, 0.02, 1e-4, 5, 3)      # n_iter k0 cooling c_rep rel_eps window freq


@pytest.fixture(scope="module")
def shim_cpu(tmp_path_factory):
    from conftest import build_r_shim_harness
    return build_r_shim_harness(str(tmp_path_factory.mktemp("shim") / "harness_cpu"), real_library=False)


@pytest.fixture
def problem_bin(tmp_path):
    from conftest import write_problem_bin
    hold = (np.array([0, 3, 7], np.int32), np.array([5, 9, 11], np.int32), np.array([1.5, 2.5, 0.25]))
    write_problem_bin(tmp_path / "p.bin", *small_problem(50, 4, 0.2, 3), hold)
    return tmp_path / "p.bin"


def _harness(exe, *args):
    out = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


def _modes(exe, problem_bin, out, keep, *modes):
    return _harness(exe, "batch_modes", problem_bin, out, len(modes), *BATCH_ARGS, keep, *modes)


@pytest.mark.parametrize("keep", [1, 0])
def test_eleventh_element_sets_the_mode_of_its_job(shim_cpu, problem_bin, tmp_path, keep):
    r = _modes(shim_cpu, problem_bin, tmp_path / "m.bin", keep, "rowblock", "-", "coloured", "rowblock")
    assert r["left_by"] == "return" and r["protect_depth"] == 0 and r["type_errors"] == 0 and r["errors"] == 0
    got = [int(j["message"].split("mode=")[1].split()[0]) for j in r["jobs"]]
    assert got == [_lib.MODE_ROWBLOCK, _lib.MODE_COLOURED, _lib.MODE_COLOURED, _lib.MODE_ROWBLOCK]
    assert all(j["status"] == 0 for j in r["jobs"])
    assert all(j["pos_len"] == (50 * 4 if keep else 0) for j in r["jobs"])


def test_jobs_of_ten_elements_are_the_plain_batch(shim_cpu, problem_bin, tmp_path):
    a = _harness(shim_cpu, "batch", problem_bin, tmp_path / "a.bin", 3, *BATCH_ARGS, 1)
    b = _modes(shim_cpu, problem_bin, tmp_path / "b.bin", 1, "-", "-", "-")
    a.pop("scenario"), b.pop("scenario")
    assert a == b
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "b.bin").read_bytes()


@pytest.mark.parametrize("bad", ["replay", "Rowblock", "", "NA", "@int", "@real"])
def test_bad_mode_is_an_r_error_naming_the_job(shim_cpu, problem_bin, tmp_path, bad):
    r = _modes(shim_cpu, problem_bin, tmp_path / "m.bin", 1, "coloured", bad, "rowblock")
    assert r["left_by"] == "Rf_error" and r["errors"] == 1 and r["protect_depth"] == 0 and r["type_errors"] == 0
    assert r["message"].startswith("job 2:") and "mode" in r["message"]
    assert r["interrupt_checks"] == 0                  # the library was not called


# ---- cv / sampler: `mode` reaches every job of the batch ----
def _recording_fit_batch(seen):
    def stub(jobs, device=0, **kw):
        seen.append([j.get("mode") for j in jobs])
        return [dict(status=_lib.OK, holdout_sum_abs=1.0, holdout_count=2, iterations=3, converged=True) for _ in jobs]
    return stub


@pytest.mark.parametrize("mode,code", [("coloured", _lib.MODE_COLOURED), ("rowblock", _lib.MODE_ROWBLOCK)])
def test_cv_entries_pass_the_mode_to_every_job(monkeypatch, mode, code):
    seen = []
    monkeypatch.setattr(_lib, "fit_batch", _recording_fit_batch(seen))
    m = random_r_matrix(24, 0.6, 3)
    samples = [dict(N=2, k0=1.0, cooling_rate=0.01, c_repulsion=0.01), dict(N=20, k0=2.0, cooling_rate=0.02, c_repulsion=0.01)]
    cv.likelihood_batch(m, samples, 5, 1e-4, folds=3, mode=mode)
    cv.likelihood_function(m, 5, 1e-4, 20, 1.0, 0.01, 0.01, folds=3, mode=mode)
    rows, cols = np.triu_indices(24, 1)
    vals = np.array([m[r, c] for r, c in zip(rows, cols)], dtype=object)
    keep = np.array([v is not None for v in vals])
    cv.likelihood_batch_coo(24, rows[keep], cols[keep], vals[keep], samples, 5, 1e-4, folds=3, mode=mode)
    assert len(seen) == 3 and all(len(s) > 0 and all(x == code for x in s) for s in seen), seen


def test_cv_default_mode_is_coloured_and_unknown_modes_are_refused(monkeypatch):
    seen = []
    monkeypatch.setattr(_lib, "fit_batch", _recording_fit_batch(seen))
    m = random_r_matrix(20, 0.6, 4)
    cv.likelihood_batch(m, [dict(N=2, k0=1.0, cooling_rate=0.01, c_repulsion=0.01)], 5, 1e-4, folds=2)
    assert seen and all(x == _lib.MODE_COLOURED for x in seen[0])
    for bad in ("replay", "row-block"):
        with pytest.raises(ValueError, match="mode"):
            cv.likelihood_batch(m, [dict(N=2, k0=1.0, cooling_rate=0.01, c_repulsion=0.01)], 5, 1e-4, folds=2, mode=bad)


def test_adaptive_mc_batch_passes_the_mode(monkeypatch):
    seen = []
    monkeypatch.setattr(_lib, "fit_batch", _recording_fit_batch(seen))
    rng = np.random.default_rng(5)
    table = {"log_N": np.log(rng.uniform(17, 30, 12)), "log_k0": rng.normal(0, 1, 12), "log_cooling_rate": rng.normal(-4, 1, 12),
             "log_c_repulsion": rng.normal(-4, 1, 12), "NLL": rng.uniform(10, 20, 12), "Holdout_MAE": rng.uniform(1, 2, 12)}
    m = random_r_matrix(24, 0.6, 6)
    sampler.adaptive_mc_batch(table, m, 2, 3, 5, 1e-4, folds=2, rng=rng, mode="rowblock")
    assert len(seen) == 2 and all(len(s) > 0 and all(x == _lib.MODE_ROWBLOCK for x in s) for s in seen)
