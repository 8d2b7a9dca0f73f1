"""Tensor-parallel SwiGLU MLP (Megatron column->row) on the fused sm_100a ops.

API mirrors /root/reference/python/triton_dist/layers/nvidia/tp_mlp.py:52-270 (``_init_parameters``, ``_init_ctx``,
``torch_fwd``, ``dist_triton_fwd`` = ag_gemm -> silu*mul -> gemm_rs, ``dist_triton_AR_fwd``,
``dist_triton_gemm_ar_fwd`` + the micro-bench helpers).  Differences: the activation is one fused CUDA kernel
and the non-fused GEMMs also run on our tcgen05 kernel (the reference calls cuBLAS through F.linear there).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist

from .. import utils as U
from ..ops import comm
from ..ops.ag_gemm import ag_gemm, ag_gemm_mxfp8, create_ag_gemm_context
from ..ops.elementwise import silu_mul
from ..ops.gemm import gemm
from ..ops.gemm_ar import create_gemm_ar_context_auto, low_latency_gemm_allreduce_op
from ..ops.fp8 import quantize_mxfp8
from ..ops.gemm_rs import create_gemm_rs_context, gemm_rs, gemm_rs_mxfp8


def shard_local(tensor: torch.Tensor, world_size: int, dim: int, local_rank: int) -> torch.Tensor:
    if tensor.shape[dim] % world_size:
        raise ValueError(f"dimension {dim} of size {tensor.shape[dim]} is not divisible by world size {world_size}")
    return tensor.split(tensor.shape[dim] // world_size, dim=dim)[local_rank].contiguous()


def _linear(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """``x @ w.T`` on the tcgen05 kernel (GPU) or eager (emulation)."""
    if x.is_cuda:
        return gemm(x, w)
    return torch.nn.functional.linear(x, w)


class TP_MLP:
    def __init__(self, rank: int = 0, world_size: int = 8, group=None):
        self.rank, self.world_size, self.group = rank, world_size, group
        self.gate_up_proj: Optional[torch.Tensor] = None   # [2 * I / W, H]
        self.down_proj: Optional[torch.Tensor] = None      # [H, I / W]
        self.ag_ctx = self.rs_ctx = self.ar_ctx = self.gemm_ar_ctx = None
        self.ar_method = comm.AllReduceMethod.Unknown
        self.gate_up_mx = self.down_mx = None               # MXFP8 weights of dist_triton_mxfp8_fwd

    # ---- parameters -------------------------------------------------------------------------------------
    def _init_parameters(self, mlp, verbose: bool = False):
        """``mlp``: any module with ``gate_proj / up_proj / down_proj`` Linear children (HF layout)."""
        dev = U.current_device()
        gate = shard_local(mlp.gate_proj.weight.detach(), self.world_size, 0, self.rank)
        up = shard_local(mlp.up_proj.weight.detach(), self.world_size, 0, self.rank)
        self.gate_up_proj = torch.cat((gate, up), dim=0).to(dev)
        self.down_proj = shard_local(mlp.down_proj.weight.detach(), self.world_size, 1, self.rank).to(dev)
        self._finish_init()

    def _init_parameters_from_shards(self, gate_up: torch.Tensor, down: torch.Tensor):
        """Already-sharded weights (random-init demo path: no full model is ever materialised)."""
        self.gate_up_proj, self.down_proj = gate_up, down
        self._finish_init()

    def _finish_init(self):
        self.ag_N_per_rank, self.K = self.gate_up_proj.shape
        self.dtype = self.gate_up_proj.dtype

    # ---- contexts -----------------------------------------------------------------------------------------
    def _init_ctx(self, max_M: int, ag_intranode_stream=None, ag_internode_stream=None, mxfp8: bool = False):
        """``mxfp8=True``: contexts for :meth:`dist_triton_mxfp8_fwd` (e4m3 all-gather workspace with its block scales) and the
        gate/up and down weights quantised to MXFP8 once, here; :meth:`dist_triton_fwd` then needs a context of its own."""
        ag_dtype = torch.float8_e4m3fn if mxfp8 else self.dtype
        self.ag_ctx = create_ag_gemm_context(max_M, self.ag_N_per_rank, self.K, ag_dtype, self.rank, self.world_size)
        self.rs_ctx = create_gemm_rs_context(max_M, self.K, self.rank, self.world_size, self.world_size,
                                             torch.bfloat16 if mxfp8 else self.dtype)
        if mxfp8:
            self.gate_up_mx = quantize_mxfp8(self.gate_up_proj)
            self.down_mx = quantize_mxfp8(self.down_proj)
        U.barrier_all_host()

    def _init_AR_ctx(self, max_M: int, method=comm.AllReduceMethod.Unknown, dtype=torch.bfloat16):
        self.ar_method = method
        N = self.down_proj.shape[0]
        self.ar_ctx = comm.create_allreduce_ctx(max_M * N * torch.empty(0, dtype=dtype).element_size(), self.rank,
                                                self.world_size, self.world_size)

    def _init_gemm_ar_ctx(self, max_M: int, dtype=torch.bfloat16):
        self.gemm_ar_ctx = create_gemm_ar_context_auto(self.rank, self.world_size, max_M, self.down_proj.shape[0], dtype)

    def finalize(self):
        for c in (self.ag_ctx, self.rs_ctx, self.ar_ctx, self.gemm_ar_ctx):
            if c is not None:
                c.finalize()
        self.ag_ctx = self.rs_ctx = self.ar_ctx = self.gemm_ar_ctx = None

    # ---- forwards -----------------------------------------------------------------------------------------
    @torch.inference_mode()
    def torch_fwd(self, x: torch.Tensor) -> torch.Tensor:
        """Baseline: cuBLAS + NCCL all-reduce (what the fused paths are compared against)."""
        out = torch.nn.functional.linear(x, self.gate_up_proj)
        wg, w1 = torch.chunk(out, 2, dim=-1)
        out = torch.nn.functional.linear(torch.nn.functional.silu(wg) * w1, self.down_proj)
        if self.world_size > 1:
            dist.all_reduce(out, group=self.group)
        return out

    @torch.inference_mode()
    def dist_triton_fwd(self, x: torch.Tensor, autotune: bool = False) -> torch.Tensor:
        """AG-GEMM -> fused SiLU*up -> GEMM-RS.  ``x``: this rank's rows ``[M/W, H]`` -> ``[M/W, H]``."""
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        h = ag_gemm(x2, self.gate_up_proj.t(), self.ag_ctx)
        h = silu_mul(h)
        out = gemm_rs(h, self.down_proj.t(), self.rs_ctx)
        return out.view(*shp[:-1], -1) if len(shp) == 3 else out

    @torch.inference_mode()
    def dist_triton_mxfp8_fwd(self, x: torch.Tensor) -> torch.Tensor:
        """MXFP8 TP MLP (contexts from ``_init_ctx(..., mxfp8=True)``): quantise x -> AG-GEMM on e4m3 rows + block scales ->
        fused SiLU*up -> quantise -> GEMM-RS, bf16 out.  ``x``: this rank's rows ``[M/W, H]`` (``M/W % 128 == 0``)."""
        if self.gate_up_mx is None:
            raise RuntimeError("dist_triton_mxfp8_fwd needs _init_ctx(max_M, mxfp8=True)")
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        h = ag_gemm_mxfp8(quantize_mxfp8(x2), self.gate_up_mx, self.ag_ctx)
        h = silu_mul(h)
        out = gemm_rs_mxfp8(quantize_mxfp8(h), self.down_mx, self.rs_ctx)
        return out.view(*shp[:-1], -1) if len(shp) == 3 else out

    @torch.inference_mode()
    def dist_triton_AR_fwd(self, x: torch.Tensor) -> torch.Tensor:
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        h = silu_mul(_linear(x2, self.gate_up_proj))
        out = _linear(h, self.down_proj)
        if self.world_size > 1:
            out = comm.all_reduce(out.contiguous(), self.ar_method, self.ar_ctx)
        return out.view(shp)

    @torch.inference_mode()
    def dist_triton_gemm_ar_fwd(self, x: torch.Tensor) -> torch.Tensor:
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        h = silu_mul(_linear(x2, self.gate_up_proj))
        out = low_latency_gemm_allreduce_op(self.gemm_ar_ctx, h, self.down_proj)
        return out.view(shp)

    def fwd(self, x):
        raise NotImplementedError("use torch_fwd / dist_triton_fwd / dist_triton_AR_fwd / dist_triton_gemm_ar_fwd")

    # ---- micro-bench helpers (tp_mlp.py:227-270) -------------------------------------------------------------
    @torch.inference_mode()
    def torch_ag_gemm(self, x):
        M = x.shape[0] * self.world_size
        buf = torch.empty((M, x.shape[1]), dtype=x.dtype, device=x.device)
        dist.all_gather_into_tensor(buf, x, group=self.group)
        return torch.matmul(buf, self.gate_up_proj.t())

    @torch.inference_mode()
    def dist_triton_ag_gemm(self, x, autotune: bool = False):
        return ag_gemm(x, self.gate_up_proj.t(), self.ag_ctx)

    @torch.inference_mode()
    def torch_gemm_rs(self, x):
        out = torch.matmul(x, self.down_proj.t())
        rs = torch.empty((x.shape[0] // self.world_size, out.shape[1]), dtype=x.dtype, device=x.device)
        dist.reduce_scatter_tensor(rs, out, group=self.group)
        return rs

    @torch.inference_mode()
    def dist_triton_gemm_rs(self, x, autotune: bool = False):
        return gemm_rs(x, self.down_proj.t(), self.rs_ctx)
