"""8-bit AllGather + GEMM without a GPU: the int8 / e4m3 / MXFP8 cases on the shared-memory emulation backend (8-bit rows and their
scales move through the heap workspace under the flag protocol and are dequantised by the consumer), the rejected combinations,
and what the sm_100a cross-compile made of the kAG kernels."""
import os
import re
import shutil
import subprocess

import pytest

from ag_gemm_q8_worker import run_cases

CPU_ENV = {"TD_FORCE_HOST_BACKEND": "1", "CUDA_VISIBLE_DEVICES": ""}
CASES = ["ag_gemm_q8", "ag_gemm_q8_reject", "tp_mlp_mxfp8"]


@pytest.mark.parametrize("world", [2, 3])
def test_ag_gemm_q8_emulated(world):
    run_cases(CASES, nproc=world, env_extra=CPU_ENV, timeout=900)


def _cuobjdump():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    from triton_dist import _build
    return exe, str(_build.build_cuda())


def test_kag_kernels_carry_8bit_mma_and_do_not_spill():
    """Every kAG instantiation of the tcgen05 GEMM (mode 1) holds the MMA of the kinds it serves: the 16-bit-layout ones run bf16,
    int8 (UTCIMMA) and e4m3 (UTCQMMA); the MXFP8 ones the block-scaled UTCQMMA.  No GEMM kernel uses local memory (spills)."""
    exe, lib = _cuobjdump()
    sass = subprocess.run([exe, "-sass", lib], capture_output=True, text=True, check=True).stdout
    mmas, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"\b(UTC[A-Z]*MMA)", line)
        if cur and m and "gemm_kernelILi1E" in cur:
            mmas.setdefault(cur, set()).add(m.group(1))
    fp8 = [k for k in mmas if re.search(r"ELb1E", k)]
    q8 = [k for k in mmas if re.search(r"ELb0E", k)]
    assert len(fp8) == 4 and len(q8) >= 10, sorted(mmas)
    for k in fp8:
        assert mmas[k] == {"UTCQMMA"}, (k, mmas[k])
    for k in q8:
        assert {"UTCHMMA", "UTCIMMA", "UTCQMMA"} <= mmas[k], (k, mmas[k])
    res = subprocess.run([exe, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    usage = re.findall(r"Function (\S*gemm_kernel\S*):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", res)
    assert usage, res[:2000]
    spills = [(f, st, lo) for f, _, st, lo in usage if st != "0" or lo != "0"]
    assert not spills, spills
