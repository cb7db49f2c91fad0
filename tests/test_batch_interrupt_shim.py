"""CPU tests of the interruptible batch .Call (integration/r_shim.c -> topolow_fit_batch_interruptible) against the
recording fake of the library (integration/r_stub/fake_topolow.c), which polls once before each job."""
import json
import subprocess

import numpy as np
import pytest

from conftest import small_problem

BATCH_ARGS = (250, 4.0, 0.01, 0.02, 1e-4, 5, 3, 1)      # n_iter k0 cooling c_rep rel_eps window freq keep


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


@pytest.mark.parametrize("k", [1, 2, 5])
def test_batch_interrupt_leaves_through_the_shim(shim_cpu, problem_bin, tmp_path, k):
    # the interrupt is caught inside R_ToplevelExec and reported to the library; the library returns
    # TOPOLOW_ERR_INTERRUPTED and the shim raises the R condition from its own frame, with the protect stack unwound
    r = _harness(shim_cpu, "batch_interrupt", problem_bin, tmp_path / "o.bin", 5, *BATCH_ARGS, k)
    assert r["left_by"] == "Rf_onintr" and r["onintr_calls"] == 1 and r["interrupt_checks"] == k
    assert r["raw_interrupt_jumps"] == 0 and r["protect_depth"] == 0 and r["errors"] == 0


def test_batch_interrupt_without_interrupt_equals_batch(shim_cpu, problem_bin, tmp_path):
    a = _harness(shim_cpu, "batch", problem_bin, tmp_path / "a.bin", 5, *BATCH_ARGS)
    b = _harness(shim_cpu, "batch_interrupt", problem_bin, tmp_path / "b.bin", 5, *BATCH_ARGS, 0)
    assert b["left_by"] == "return" and b["interrupt_checks"] == 5 and b["onintr_calls"] == 0
    assert "shared=4" in b["jobs"][0]["message"]
    a.pop("scenario"), b.pop("scenario")
    assert a == b
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "b.bin").read_bytes()
