"""CPU test of the built library's resource usage (cuobjdump -res-usage): the spring walk runs beside the two-GEMM
repulsion pass only while two pass CTAs and one walk CTA fit in an SM's registers and shared memory
(rowblock.cu: launch_iteration, the static_assert next to kWalkSmem).  One register more in either kernel brings back
the serial walk without any other symptom than the time per iteration, so the caps are checked for every H."""
import os
import re
import shutil
import subprocess

import pytest

from topolow_b200 import _lib

REGS_PER_SM = 65536
WALK_THREADS, WALK_REGS = 128, 112         # kBlockRows, kWalkRegs
PASS_THREADS, PASS_REGS = 320, 80          # kT2Threads, __maxnreg__ of repulse_tc2_kernel
WALK_SHARED = 1152                         # kWalkStaticSmem: static shared memory + the 1 KiB reserve, as cuobjdump reports it
H_VALUES = range(1, 9)                     # ndim 1..16


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")):
        if cand and os.path.exists(cand):
            return cand
    return None


@pytest.fixture(scope="module")
def usage():
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump (CUDA toolkit) not found")
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    out = subprocess.run([tool, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    res = {}
    for name, regs, shared in re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:\d+ SHARED:(\d+)", out):
        res[name] = (int(regs), int(shared))
    return res


def _kernels(usage, pattern):
    return {n: v for n, v in usage.items() if re.search(pattern, n)}


def test_walk_and_pass_register_budget(usage):
    assert WALK_THREADS * WALK_REGS + 2 * PASS_THREADS * PASS_REGS <= REGS_PER_SM
    for h in H_VALUES:
        walk = _kernels(usage, r"spring_kernelILi%dELi\d+E" % h)
        assert len(walk) == 2, f"spring_kernel<{h}, *>: expected the 4- and 8-deep rings, found {sorted(walk)}"
        for name, (regs, shared) in walk.items():
            assert regs <= WALK_REGS, f"{name}: {regs} registers > {WALK_REGS}"
            assert shared <= WALK_SHARED, f"{name}: {shared} bytes of static shared memory > {WALK_SHARED}"
        rep = _kernels(usage, r"repulse_tc2_kernelILi%dEE" % h)
        assert len(rep) == 1, f"repulse_tc2_kernel<{h}>: found {sorted(rep)}"
        for name, (regs, _shared) in rep.items():
            assert regs <= PASS_REGS, f"{name}: {regs} registers > {PASS_REGS}"


def test_repulsion_kernels_are_the_two_forms_the_policy_runs(usage):
    """For every H of ndim 1..16 the library holds the kernels of the two forms of the repulsion pass and nothing else:
    one shape of the FP32 difference form (repulse_kernel) and the two-GEMM tensor-core form (image_tc_kernel,
    repulse_tc2_kernel)."""
    for h in H_VALUES:
        found = sorted(re.search(r"((?:repulse|image)\w*?)ILi", n).group(1)
                       for n in _kernels(usage, r"(?:repulse|image)\w*?ILi%dE" % h))
        assert found == ["image_tc_kernel", "repulse_kernel", "repulse_tc2_kernel"], f"H = {h}: {found}"
