"""CPU checks of the row-block mode at ndim 17..32.

The built library (cuobjdump -res-usage) holds, for every H of that range (10, 12, 14, 16), the kernels the mode launches
- spring and MAE walks with both ring depths, combine_kernel, the FP32 difference form of the repulsion pass - with no
stack (no spills) and within the register caps of rowblock.cu, and not the tensor-core form, which exists for
ndim <= 16 only.  And the FP64 restatement shows the invariant the padded rows rely on: zero columns stay zero
and leave the other columns bit for bit as they are."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import small_problem
from oracle import cpu_oracle
from topolow_b200 import _lib, rowblock

H_WIDE = (10, 12, 14, 16)       # ndim 17..32: H = Dp / 2, Dp = ndim rounded up to a multiple of 4
WALK_REGS_WIDE = 168            # kWalkRegsWide
REP_REGS_WIDE = 128             # kRepRegsWide
MAE_REGS, COMBINE_REGS = 128, 128


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
    return {name: (int(regs), int(stack))
            for name, regs, stack in re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)}


def _kernels(usage, pattern):
    return {n: v for n, v in usage.items() if re.search(pattern, n)}


@pytest.mark.parametrize("h", H_WIDE)
def test_wide_rows_launched_kernels_exist_without_spills_within_their_caps(usage, h):
    for kernel, count, cap in ((r"spring_kernelILi%dELi\d+E", 2, WALK_REGS_WIDE), (r"mae_kernelILi%dELi\d+E", 2, MAE_REGS),
                               (r"combine_kernelILi%dEE", 1, COMBINE_REGS),
                               (r"repulse_kernelILi%dELi1ELi\d+ELi%dEE", 1, REP_REGS_WIDE)):
        pat = kernel % ((h, REP_REGS_WIDE) if "repulse" in kernel else h)
        found = _kernels(usage, pat)
        assert len(found) == count, f"{pat}: expected {count}, found {sorted(found)}"
        for name, (regs, stack) in found.items():
            assert stack == 0, f"{name}: {stack} bytes of stack"
            assert regs <= cap, f"{name}: {regs} registers > {cap}"


@pytest.mark.parametrize("h", H_WIDE)
def test_wide_rows_build_no_tensor_or_inner_product_form(usage, h):
    for kernel in ("repulse_tc2_kernel", "image_tc_kernel"):
        found = _kernels(usage, r"%sILi%dE" % (kernel, h))
        assert not found, sorted(found)
    # only the one shape of the difference form
    assert len(_kernels(usage, r"repulse_kernelILi%dE" % h)) == 1


def test_zero_columns_leave_the_others_bit_identical():
    n = 500
    init18, deg, ei, ej, ed, et = small_problem(n, 18, 0.1, 1820, thresholds=True)
    init20 = np.hstack([init18, np.zeros((n, 2))])
    hp = (12, 5.0, 0.01, 0.02, 1e-4, 5, 3)
    sop = rowblock.slot_order(n)
    a = cpu_oracle.relaxed_optimize_layout(init18, deg, ei, ej, ed, et, *hp, seed=4, slot_of_point=sop, trace=True)
    b = cpu_oracle.relaxed_optimize_layout(init20, deg, ei, ej, ed, et, *hp, seed=4, slot_of_point=sop, trace=True)
    assert np.array_equal(b["positions"][:, :18], a["positions"])
    assert not np.any(b["positions"][:, 18:])
    assert b["final_mae"] == a["final_mae"] and b["iterations"] == a["iterations"]
    assert np.array_equal(b["trace_mae"], a["trace_mae"], equal_nan=True)
