"""Resources of the tcgen05 GMM-drift integrator K1-T (csrc/integrator_tc.cu), checked at compile time.

The kinetic instances keep the code they had before the overdamped switch was added: the same register count and the
same SASS, function by function (a digest of the instruction text, addresses and encodings stripped, taken from the
build before the switch with CUDA 12.9; the digest comparison is skipped under another compiler release).  The
overdamped instances (K1-T-OD) compile without spills or stack and keep the tcgen05 GEMMs (UTCHMMA) and their TMEM
loads (LDTM) in their SASS.
"""
import hashlib
import os
import re
import shutil
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pde_inverse_problem_b200", "csrc")

# (d, KP, BLK, MINB) -> (registers, SASS digest) of the kinetic instances
KINETIC = {
    (8, 16, False, 6): (76, "839f146004ea159c"),
    (8, 16, False, 8): (62, "7e9080ffba188d17"),
    (8, 16, True, 6): (79, "92a509d770f44134"),
    (8, 16, True, 8): (64, "2a8f741a8a2792bc"),
    (8, 32, False, 6): (78, "15945549452bc96c"),
    (8, 32, False, 8): (64, "214f074c47777e28"),
    (8, 32, True, 6): (80, "db48b079669ecb30"),
    (8, 32, True, 8): (64, "44afefa641bddae9"),
    (8, 48, False, 6): (80, "7b4cde5a3ff0ef3c"),
    (8, 48, False, 8): (64, "3dbf25bc449aa87a"),
    (8, 48, True, 6): (80, "cf42a8f1ff7fb680"),
    (8, 48, True, 8): (64, "8cdb49a0a61c1f33"),
    (8, 64, False, 6): (80, "043953e173f8a326"),
    (8, 64, False, 8): (64, "2e360ee56ffc0bfb"),
    (8, 64, True, 6): (80, "9d91e6fdbadf1920"),
    (8, 64, True, 8): (64, "d35cf7fd5adf5e20"),
    (16, 16, False, 3): (108, "cd095e11b5bd55fc"),
    (16, 16, False, 4): (103, "0cc9362cfb6b3573"),
    (16, 16, True, 3): (94, "7a818598a8efdd8b"),
    (16, 16, True, 4): (102, "955134152f10f51c"),
    (16, 32, False, 3): (128, "10e5a4bea9def6f2"),
    (16, 32, False, 4): (120, "6def6a7f4536b5d6"),
    (16, 32, True, 3): (114, "95311dd2854fd64e"),
    (16, 32, True, 4): (118, "9a31b848c99dbf79"),
    (16, 48, False, 3): (135, "2907f0ffbc180d10"),
    (16, 48, False, 4): (126, "61a5690bdcf72616"),
    (16, 48, True, 3): (128, "7e19d9610a3027d6"),
    (16, 48, True, 4): (128, "9a395842402a3ab2"),
    (16, 64, False, 3): (151, "008858d2ae472b00"),
    (16, 64, False, 4): (126, "3f8eb6b98425f938"),
    (16, 64, True, 3): (146, "e93ae2b37c9f7742"),
    (16, 64, True, 4): (128, "02cb6972723c9f29"),
    (32, 16, False, 3): (158, "0cf9f4fb2bfeee67"),
    (32, 16, False, 4): (124, "bb52591e9271a36d"),
    (32, 16, True, 3): (128, "64ffb0abb4bcb2c5"),
    (32, 16, True, 4): (124, "dc50aa5889a0fc71"),
    (32, 32, False, 3): (156, "36d1197d0aefbc68"),
    (32, 32, False, 4): (128, "d4e061b80810b76b"),
    (32, 32, True, 3): (144, "33d7906f3d8ba545"),
    (32, 32, True, 4): (128, "00dd2016a604db8a"),
    (32, 48, False, 3): (156, "65bd44d016629637"),
    (32, 48, False, 4): (128, "dfe4d83cd8e2fe02"),
    (32, 48, True, 3): (164, "d48519da4f27d872"),
    (32, 48, True, 4): (128, "afcdfb6b6e7247f0"),
    (32, 64, False, 3): (168, "d74a14a5d7da3d4c"),
    (32, 64, False, 4): (128, "9782c696ec44ae74"),
    (32, 64, True, 3): (168, "22e9b03cbb33a7d4"),
    (32, 64, True, 4): (128, "a28adea700414c35"),
}
DIGEST_RELEASE = "release 12.9"
# the overdamped instances: (d, KP, mode) with mode 0 = terminal only, 1 = BLOCK128, 2 = TIME_SOA
OD = {(d, kp, mode) for d in (8, 16, 32) for kp in (16, 32, 48, 64) for mode in (0, 1, 2)}


def _tool(name):
    return shutil.which(name) or next((p for p in (f"/usr/local/cuda/bin/{name}",) if os.path.exists(p)), None)


def _key(mangled):
    """(kinetic?, key) of a kl_integrate_tc*_kernel instance from its mangled name, None for other functions"""
    m = re.search(r"kl_integrate_tc(8?)_kernelILi(\d+)E(?:Li(\d+)E)?Lb([01])ELi(\d+)ELb([01])ELb([01])E", mangled)
    if not m:
        return None
    d, kp = (8, int(m.group(2))) if m.group(1) else (int(m.group(2)), int(m.group(3)))
    blk, minb, od, traj = m.group(4) == "1", int(m.group(5)), m.group(6) == "1", m.group(7) == "1"
    if od:
        return False, (d, kp, 0 if not traj else (1 if blk else 2))
    return True, (d, kp, blk, minb)


@pytest.fixture(scope="module")
def report():
    nvcc, cuobjdump = _tool("nvcc"), _tool("cuobjdump")
    if nvcc is None or cuobjdump is None:
        pytest.skip("nvcc / cuobjdump not found")
    release = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "itc.o")
        cmd = [nvcc, "-O3", "-std=c++17", "-DPDEIP_HAVE_TENSOR_PATH", "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC, "--expt-relaxed-constexpr",
               "-Xptxas", "-v", "-c", os.path.join(CSRC, "integrator_tc.cu"), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
        sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = _key(m.group(1))
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
            k = _key(m.group(1))
            body = out.setdefault(k, {}) if k else None
            if body is not None:
                body["ins"], body["ops"] = [], set()
            continue
        if body is None:
            continue
        m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m:
            body["ins"].append(m.group(1).strip())
            body["ops"].update(op for op in ("UTCHMMA", "LDTM") if op in line)
    for r_ in out.values():
        r_["digest"] = hashlib.sha256("\n".join(r_.pop("ins", [])).encode()).hexdigest()[:16]
    return out, DIGEST_RELEASE in release


def test_every_instance_reported(report):
    out, _ = report
    want = {(True, k) for k in KINETIC} | {(False, k) for k in OD}
    assert set(out) == want, sorted(set(out) ^ want)


@pytest.mark.parametrize("inst", sorted(KINETIC))
def test_kinetic_instances_unchanged(report, inst):
    out, same_release = report
    r = out[(True, inst)]
    regs, digest = KINETIC[inst]
    assert r["regs"] == regs, (inst, r)
    if same_release:
        assert r["digest"] == digest, (inst, r["digest"])


@pytest.mark.parametrize("inst", sorted(OD))
def test_overdamped_instances_no_spills_and_tcgen05(report, inst):
    r = report[0][(False, inst)]
    assert r["spill"] == 0 and r["stack"] == 0, (inst, r)
    assert r["ops"] == {"UTCHMMA", "LDTM"}, (inst, r["ops"])
