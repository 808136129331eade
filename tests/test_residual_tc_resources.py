"""Register budget of the tcgen05 residual kernels (csrc/residual_tensor.cu), checked at compile time.

The kernels move registers between warpgroups with `setmaxnreg`: the epilogue warps grow into what the idle warps of the
extra warpgroup release, and that pool is set by the register count the kernel is LAUNCHED at.  A `setmaxnreg` request
the pool cannot serve never returns (the kernel hangs), so the count ptxas reports must be the one the Regs budget
assumes (Team<NS>::kLaunchRegs: 168 for the two-slot d = 8 kernel at 384 threads, 96 for the one-slot kernels at 640).
Spill stores are held at or below their measured figures (each a few words of loop state; none in the epilogue phases).
"""
import os
import re
import shutil
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pde_inverse_problem_b200", "csrc")

LAUNCH_REGS = {1: 96, 2: 168}
# (DP, NS, MODE) -> spill-store bytes allowed; MODE 0 KFP 0T, 1 KFP boundary, 2 FP 0T
MAX_SPILL = {(32, 1, 0): 0, (32, 1, 1): 0, (32, 1, 2): 8,
             (16, 1, 0): 0, (16, 1, 1): 0, (16, 1, 2): 0,
             (8, 2, 0): 0, (8, 2, 1): 0, (8, 2, 2): 12}


def _nvcc():
    return shutil.which("nvcc") or next((p for p in ("/usr/local/cuda/bin/nvcc",) if os.path.exists(p)), None)


@pytest.fixture(scope="module")
def ptxas_report():
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-O3", "-std=c++17", "-DPDEIP_HAVE_TENSOR_PATH", "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC, "--expt-relaxed-constexpr",
               "-Xptxas", "-v", "-c", os.path.join(CSRC, "residual_tensor.cu"), "-o", os.path.join(tmp, "rt.o")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    out = {}
    cur = None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            k = re.search(r"mlp_residual_tc_kernelILi(\d+)ELi(\d+)ELi(\d+)E", m.group(1))
            cur = tuple(int(x) for x in k.groups()) if k else None
            if cur:
                out[cur] = {}
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores", line)
        if m:
            out[cur]["spill"] = int(m.group(1))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out[cur]["regs"] = int(m.group(1))
    return out


def test_every_instance_reported(ptxas_report):
    assert set(ptxas_report) == set(MAX_SPILL), sorted(ptxas_report)


@pytest.mark.parametrize("inst", sorted(MAX_SPILL))
def test_launch_registers_match_budget(ptxas_report, inst):
    assert ptxas_report[inst]["regs"] == LAUNCH_REGS[inst[1]], (inst, ptxas_report[inst])


@pytest.mark.parametrize("inst", sorted(MAX_SPILL))
def test_spill_stores_bounded(ptxas_report, inst):
    assert ptxas_report[inst]["spill"] <= MAX_SPILL[inst], (inst, ptxas_report[inst])
