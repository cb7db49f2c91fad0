"""CPU tests of the multi-device batch: the .Call shim (integration/r_shim.c) with a vector `device` against the recording
fake of the library (integration/r_stub/fake_topolow.c), the C-ABI export, and the no-GPU path of the real library."""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, has_cuda, small_problem
from topolow_b200 import _lib

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


def _devices(exe, problem_bin, out, kind, *devices):
    return _harness(exe, "batch_devices", problem_bin, out, 5, *BATCH_ARGS, kind, *devices)


@pytest.mark.parametrize("kind", ["int", "double"])
def test_device_vector_reaches_the_multi_device_entry(shim_cpu, problem_bin, tmp_path, kind):
    r = _devices(shim_cpu, problem_bin, tmp_path / "d.bin", kind, 0, 1, 3, 1)
    assert r["left_by"] == "return" and r["protect_depth"] == 0 and r["type_errors"] == 0 and r["errors"] == 0
    assert r["jobs"][0]["message"].endswith(" devices=0,1,3,1")
    assert r["interrupt_checks"] == 5                  # the poll callback went with it
    a = _harness(shim_cpu, "batch", problem_bin, tmp_path / "a.bin", 5, *BATCH_ARGS)
    r["jobs"][0]["message"] = r["jobs"][0]["message"][:-len(" devices=0,1,3,1")]
    for k in ("scenario", "interrupt_checks"):
        a.pop(k), r.pop(k)
    assert a == r
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "d.bin").read_bytes()


@pytest.mark.parametrize("kind", ["int", "double"])
def test_one_device_still_reaches_the_single_device_entry(shim_cpu, problem_bin, tmp_path, kind):
    a = _harness(shim_cpu, "batch_interrupt", problem_bin, tmp_path / "a.bin", 5, *BATCH_ARGS, 0)
    r = _devices(shim_cpu, problem_bin, tmp_path / "d.bin", kind, 0)
    assert "devices=" not in r["jobs"][0]["message"] and r["protect_depth"] == 0 and r["type_errors"] == 0
    a.pop("scenario"), r.pop("scenario")
    assert a == r
    assert (tmp_path / "a.bin").read_bytes() == (tmp_path / "d.bin").read_bytes()


@pytest.mark.parametrize("kind,devices", [("int", ()), ("double", ()), ("int", ("NA",)), ("double", ("NA",)),
                                          ("int", (0, "NA")), ("double", (1, "NA"))])
def test_empty_or_na_device_is_an_r_error(shim_cpu, problem_bin, tmp_path, kind, devices):
    r = _devices(shim_cpu, problem_bin, tmp_path / "d.bin", kind, *devices)
    assert r["left_by"] == "Rf_error" and r["errors"] == 1 and r["protect_depth"] == 0 and r["type_errors"] == 0
    assert "device" in r["message"]
    assert r["interrupt_checks"] == 0                  # the library was not called


def test_library_declares_and_exports_the_multi_device_entry():
    header = open(os.path.join(ROOT, "include", "topolow_b200.h")).read()
    assert re.search(r"TOPOLOW_API int topolow_fit_batch_devices\(", header)
    assert "topolow_fit_batch_devices" in _lib.EXPORTS
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert re.search(r"\bT topolow_fit_batch_devices\b", nm)
    assert hasattr(_lib.lib(), "topolow_fit_batch_devices")


def _raw_call(devices, n_jobs=2):
    """topolow_fit_batch_devices on n_jobs small jobs; returns (status, per-job statuses, first message)."""
    L = _lib.lib()
    keep = [_lib.ProblemArrays(*small_problem(30, 2, 0.3, s)) for s in range(n_jobs)]
    probs, pars, ress = (_lib.Problem * n_jobs)(), (_lib.Params * n_jobs)(), (_lib.Result * n_jobs)()
    outs = []
    for j, pa in enumerate(keep):
        probs[j] = pa.struct
        pars[j] = _lib.make_params(5, 4.0, 0.01, 0.02)[0]
        outs.append(np.zeros((pa.n, pa.ndim), order="F"))
        ress[j].positions = outs[-1].ctypes.data_as(_lib._dp)
        ress[j].status = 99
    dev = None if devices is None else (C.c_int32 * max(len(devices), 1))(*devices)
    rc = L.topolow_fit_batch_devices(n_jobs, probs, pars, ress, dev, 0 if devices is None else len(devices),
                                     _lib.INTERRUPT_FN(), None)
    return rc, [ress[j].status for j in range(n_jobs)], ress[0].message.decode()


@pytest.mark.parametrize("devices", [None, [], [-1], [0, -2]])
def test_bad_device_lists_are_refused_before_anything_runs(devices):
    rc, statuses, msg = _raw_call(devices)
    assert rc == _lib.ERR_BAD_ARG
    assert statuses == [99, 99]                        # no job was touched
    assert "device" in msg


@pytest.mark.skipif(has_cuda(), reason="checks the no-GPU failure mode")
@pytest.mark.parametrize("devices", [[0], [0, 0], [0, 1]])
def test_no_gpu_returns_err_cuda(devices):
    rc, statuses, msg = _raw_call(devices)
    assert rc == _lib.ERR_CUDA and msg
    assert statuses == [99, 99]
    jobs = [dict(initial_positions=np.zeros((3, 2)), degrees=np.ones(3, np.int32), edge_i=[0], edge_j=[1], edge_dist=[1.0],
                 edge_thresh=[0], n_iter=5, k0=4.0, cooling_rate=0.01, c_repulsion=0.02)]
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, device=devices)
    assert e.value.status == _lib.ERR_CUDA
    with pytest.raises(_lib.TopolowError) as e:
        _lib.fit_batch(jobs, device=[-1])
    assert e.value.status == _lib.ERR_BAD_ARG
