"""Resources of the tcgen05 MLP-drift integrator K1-MT (csrc/integrator_mlp_tc.cu), checked at compile time.

The kinetic instances (OD = false) keep the register counts they had before the overdamped variant was added: the
variant is a compile-time branch that leaves their code unchanged.  The overdamped instances (OD = true) compile without
spills or stack and keep the tcgen05 GEMM chain (UTCHMMA) and its TMEM loads (LDTM) in their SASS.
"""
import os
import re
import shutil
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pde_inverse_problem_b200", "csrc")

# (DP, TRAJ) -> registers of the kinetic instances (TRAJ 0 terminal only, 1 BLOCK128, 2 TIME_SOA)
KINETIC_REGS = {(32, 2): 166, (32, 1): 167, (32, 0): 161, (16, 2): 136, (16, 1): 138, (16, 0): 135,
                (8, 2): 123, (8, 1): 121, (8, 0): 119}


def _tool(name):
    return shutil.which(name) or next((p for p in (f"/usr/local/cuda/bin/{name}",) if os.path.exists(p)), None)


@pytest.fixture(scope="module")
def report():
    nvcc, cuobjdump = _tool("nvcc"), _tool("cuobjdump")
    if nvcc is None or cuobjdump is None:
        pytest.skip("nvcc / cuobjdump not found")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "imt.o")
        cmd = [nvcc, "-O3", "-std=c++17", "-DPDEIP_HAVE_TENSOR_PATH", "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC, "--expt-relaxed-constexpr",
               "-Xptxas", "-v", "-c", os.path.join(CSRC, "integrator_mlp_tc.cu"), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
        sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            k = re.search(r"kl_integrate_mlp_tc_kernelILi(\d+)ELi(\d+)ELi\d+ELb([01])E", m.group(1))
            cur = (int(k.group(1)), int(k.group(2)), k.group(3) == "1") if k else None
            if cur:
                out[cur] = {}
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            out[cur].update(stack=int(m.group(1)), spill=int(m.group(2)) + int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out[cur]["regs"] = int(m.group(1))
    body = None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            k = re.search(r"kl_integrate_mlp_tc_kernelILi(\d+)ELi(\d+)ELi\d+ELb([01])E", m.group(1))
            body = out.setdefault((int(k.group(1)), int(k.group(2)), k.group(3) == "1"), {}) if k else None
            if body is not None:
                body["sass"] = set()
            continue
        if body is not None:
            body["sass"].update(op for op in ("UTCHMMA", "LDTM") if op in line)
    return out


def test_every_instance_reported(report):
    want = {(dp, t, od) for (dp, t) in KINETIC_REGS for od in (False, True)}
    assert set(report) == want, sorted(report)


@pytest.mark.parametrize("inst", sorted(KINETIC_REGS))
def test_kinetic_instances_unchanged(report, inst):
    r = report[inst + (False,)]
    assert r["regs"] == KINETIC_REGS[inst] and r["spill"] == 0 and r["stack"] == 0, (inst, r)


@pytest.mark.parametrize("inst", sorted(KINETIC_REGS))
def test_overdamped_instances_no_spills_and_tcgen05(report, inst):
    r = report[inst + (True,)]
    assert r["spill"] == 0 and r["stack"] == 0, (inst, r)
    assert r["sass"] == {"UTCHMMA", "LDTM"}, (inst, r["sass"])
