"""8-bit AllGather + GEMM on B200s: int8 / e4m3 with per-row and per-tensor scales and MXFP8, every in-kernel transport, 1- and 2-CTA
tiles, a CUDA-graph replay and the MXFP8 TP MLP (tests/ag_gemm_q8_worker.py).  World 1 runs the
local gemm_scaled / gemm_mxfp8 path; larger worlds are skipped when the machine has too few GPUs."""
import pytest
import torch

from ag_gemm_q8_worker import run_cases

pytestmark = pytest.mark.gpu


def _ngpu():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_ag_gemm_q8_gpu(world):
    if _ngpu() < world:
        pytest.skip(f"needs >= {world} GPUs")
    cases = ["ag_gemm_q8", "ag_gemm_q8_graph", "ag_gemm_q8_reject"] + (["tp_mlp_mxfp8"] if world > 1 else [])
    run_cases(cases, nproc=world, timeout=900)
