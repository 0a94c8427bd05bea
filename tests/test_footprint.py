"""Register footprint of the gradient GEMM, read from the built library (no GPU needed).

Two CTAs of grad_tc_kernel (of different evaluations in flight) must fit on one SM, so that one streams while the
other sets up or drains: registers x threads <= 32 768, half of an SM's register file, and nothing spilled.  The
thread count is the kernel's __launch_bounds__ as recorded in the cubin, so the check follows the source.
"""
import os
import re
import shutil
import subprocess

import pytest

from kccotgan_b200 import _lib

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
KERNELS = ("grad_tc_kernel",)


def _dump(flag):
    if not os.path.isfile(_lib.LIB_PATH):
        pytest.skip("libkccot.so is not built")
    if not os.path.isfile(CUOBJDUMP):
        pytest.skip("cuobjdump not found")
    return subprocess.run([CUOBJDUMP, flag, _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout


def _res_usage():
    """{mangled name: (registers, stack bytes, local bytes)}"""
    usage, name = {}, None
    for line in _dump("-res-usage").splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.match(r"\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", line)
        if m and name:
            usage[name] = tuple(int(v) for v in m.groups())
            name = None
    return usage


def _max_threads():
    """{mangled name: threads per CTA of __launch_bounds__} from the EIATTR_MAX_THREADS of each .nv.info section"""
    out, name, want = {}, None, False
    for line in _dump("-elf").splitlines():
        if line.startswith("."):
            m = re.match(r"\.nv\.info\.(\S+)$", line)
            name, want = (m.group(1) if m else None), False
        elif name and "EIATTR_MAX_THREADS" in line:
            want = True
        elif want and line.strip().startswith("Value:"):
            x, y, z = (int(v, 16) for v in line.split()[1:4])
            out[name] = x * y * z
            want = False
    return out


def _one(table, kernel):
    found = {n: v for n, v in table.items() if re.search(rf"\d{kernel}E", n)}
    assert len(found) == 1, f"{kernel}: {sorted(found)}"
    return next(iter(found.values()))


@pytest.mark.parametrize("kernel", KERNELS)
def test_two_ctas_per_sm_fit_the_register_file(kernel):
    reg, stack, local = _one(_res_usage(), kernel)
    threads = _one(_max_threads(), kernel)
    assert reg * threads <= 32768, f"{kernel}: {reg} registers x {threads} threads"
    assert stack == 0 and local == 0, f"{kernel}: stack {stack}, local {local} bytes (spills)"
