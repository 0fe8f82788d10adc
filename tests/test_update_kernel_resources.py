"""CPU: the two TSDF update kernels compile to the resources their launch bounds promise.

Both kernels are issue-bound loops whose speed depends on how many CTAs an SM keeps resident: they are compiled with
`__launch_bounds__(kIntThreads, kIntCtasPerSm)` and must fit that many CTAs in the register file without spilling
(profiles/r2_summary.md: spilling to reach more CTAs per SM ran slower).  This reads the compiled library with
`cuobjdump`, so a source change that silently costs occupancy or adds local-memory traffic fails here, before any
GPU run."""

import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = ("integrate_kernel", "integrate_group_kernel")
REGS_PER_SM = 65536
REG_GRANULE = 8  # registers per thread are allocated in warp units of 256


def _source_constant(name):
    src = open(os.path.join(ROOT, "pyslam_b200", "csrc", "b2v_tsdf.cu")).read()
    m = re.search(rf"constexpr int {name} = (\d+);", src)
    assert m, name
    return int(m.group(1))


def _cuobjdump(*args):
    from pyslam_b200 import _lib
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    assert os.path.exists(_lib.LIB_PATH), "libb2v.so was not built"
    r = subprocess.run([exe, *args, _lib.LIB_PATH], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r.stdout


def _res_usage():
    """{kernel name: {"REG": n, "STACK": n, "LOCAL": n, ...}} for the update kernels, from cuobjdump -res-usage."""
    out = _cuobjdump("-res-usage")
    usage = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*(.*)", out):
        for k in KERNELS:
            if re.fullmatch(rf"_ZN3b2v{len(k)}{k}E.*", m.group(1)):
                usage[k] = {key: int(v) for key, v in re.findall(r"(\w+(?:\[\d+\])?):(\d+)", m.group(2))}
    return usage


def test_update_kernels_do_not_spill():
    usage = _res_usage()
    assert sorted(usage) == sorted(KERNELS), usage
    for k, u in usage.items():
        assert u["LOCAL"] == 0, f"{k} uses {u['LOCAL']} bytes of local memory (spills)"
        assert u["STACK"] == 0, f"{k} uses a {u['STACK']}-byte stack frame"
    # no spill stores or loads anywhere in the kernels' code (local-memory accesses are STL / LDL)
    sass = _cuobjdump("-sass")
    for k in KERNELS:
        m = re.search(rf"Function : _ZN3b2v{len(k)}{k}E\S*\n(.*?)(?=\n\s*Function : |\Z)", sass, flags=re.S)
        assert m, k
        assert not re.search(r"\b(STL|LDL)\b", m.group(1)), f"{k} spills to local memory"


def test_update_kernel_registers_fit_the_launch_bounds():
    threads, ctas = _source_constant("kIntThreads"), _source_constant("kIntCtasPerSm")
    usage = _res_usage()
    assert sorted(usage) == sorted(KERNELS), usage
    for k, u in usage.items():
        regs = -(-u["REG"] // REG_GRANULE) * REG_GRANULE
        assert regs * threads * ctas <= REGS_PER_SM, (
            f"{k}: {u['REG']} registers x {threads} threads leave room for fewer than {ctas} CTAs per SM")
