"""AllGather + GEMM in one kernel:  ``C[M, N/W] = allgather(A[M/W, K]) @ B[K, N/W]``.

Reference: ``create_ag_gemm_context`` / ``ag_gemm`` (/root/reference/python/triton_dist/kernels/nvidia/
allgather_gemm.py:511-619) -- there the all-gather is W-1 host-issued ``cudaMemcpyAsync`` + one
``cuStreamWriteValue`` flag per source rank (allgather.py:100-124) around a Triton persistent GEMM.

Here (csrc/gemm_sm100.cuh, mode kAG) the gather runs INSIDE the GEMM kernel.  Two in-kernel transports:

* ``sm_k`` (default): the K-sliced protocol of ``multicast`` below with unicast P2P stores to every peer (rows read once,
  one release fence per slice for all destinations) -- measured fastest on 8xB200, where ``multimem.st`` tops out near
  380 GB/s of ingress per GPU.
* ``multicast`` (NVLS): ``n_comm_ctas`` CTAs write this rank's shard ONCE
  to the multicast alias of the workspace with ``multimem.st`` -- the NVSwitch fans it out to every rank, so egress is
  1x the shard instead of (W-1)x -- K slice by K slice, publishing one flag per (source, K slice, comm CTA).  The TMA
  producer of a GEMM CTA acquires the flag of a K slice right before its first k-block, so EVERY tile starts after
  1/8 of the transfer and its mainloop follows the arrival; the tail after the last byte is one K slice + epilogue.
* ``sm`` (P2P): comm CTAs push the shard into every peer's workspace with coalesced 16-byte stores (posted writes; a
  pull design measured only ~7 GB/s per SM on 8xB200) and publish per-(source, byte slice) flags; the GEMM CTAs start
  on the local rows (tile order rotated by rank) and consume remote rows as they land.

No host barrier: workspaces are double buffered by call parity and flags carry monotone phase numbers kept on the
device.  ``copy_engine`` is the reference's host-driven transport, kept for comparison.

8-bit operands (``sm_k``, ``multicast`` and ``sm``): int8 / float8_e4m3fn shards with per-row or per-tensor ``scale_a`` travel as
8-bit rows (half the NVLink bytes of bf16) together with their fp32 per-row scales; ``ag_gemm_mxfp8`` moves e4m3 rows plus their
UE8M0 block scales.  The scales ride under the flags of the rows they belong to (csrc/gemm_sm100.cuh ``ag_push_scales``).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional

import torch

from .. import _C
from .. import utils as U
from .gemm import GemmConfig, fill_common

_CHUNK_ROWS = 128
_SUB = 8


@dataclass
class AllGatherGEMMTensorParallelContext:
    max_M: int
    N_per_rank: int
    K: int
    dtype: torch.dtype
    rank: int
    num_ranks: int
    num_local_ranks: int
    workspace: torch.Tensor = None     # symmetric [2, max_M, K]
    scale_ws: torch.Tensor = None      # 8-bit contexts: symmetric fp32 [2, max_M], gathered per-row activation scales
    sf_ws: torch.Tensor = None         # float8_e4m3fn contexts: symmetric uint8 [2, ceil(max_M / 128), K / 128, 512], MXFP8 scales
    flags: torch.Tensor = None         # symmetric int32 [2, W, 256]
    ready: torch.Tensor = None         # symmetric int32 [W]
    phase: torch.Tensor = None         # local int32 [4]
    n_comm_ctas: int = 16
    host_phase: int = 0                # emulation backend / bookkeeping mirror
    _ce_stream: object = None

    @property
    def symm_workspace(self):
        return self.workspace

    def local_input_buffer(self, rows: int) -> torch.Tensor:
        """Zero-copy entry: where the NEXT call expects my shard ([rows, K] inside the workspace).  A producer
        (e.g. the previous layer's epilogue) may write there directly and pass it as ``A``.  Host-counter based: not usable
        inside a CUDA-graph capture (the device-side parity alternates on replay)."""
        if _is_8bit(self.dtype):
            raise NotImplementedError("local_input_buffer(): zero-copy input is not supported for 8-bit ag_gemm contexts")
        if self.workspace.is_cuda and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("local_input_buffer() cannot be used while capturing a CUDA graph")
        ph = self._phase_value() + 1
        buf = self.workspace[ph & 1]
        return buf[self.rank * rows:(self.rank + 1) * rows]

    def _phase_value(self) -> int:
        return self.host_phase

    def finalize(self):
        heap = U.get_heap()
        for t in (self.workspace, self.ready, self.flags, self.scale_ws, self.sf_ws):
            if t is not None:
                heap.free_tensor(t)
        self.workspace = self.ready = self.flags = self.scale_ws = self.sf_ws = None


def create_ag_gemm_context(max_M: int, N: int, K: int, dtype: torch.dtype, rank: Optional[int] = None,
                           num_ranks: Optional[int] = None, num_local_ranks: Optional[int] = None,
                           n_comm_ctas: int = 16, BLOCK_M: Optional[int] = None, BLOCK_N: Optional[int] = None,
                           BLOCK_K: Optional[int] = None, stages: Optional[int] = None, ag_intranode_stream=None,
                           ag_internode_stream=None, for_correctness: bool = False) -> AllGatherGEMMTensorParallelContext:
    """``max_M`` = largest gathered M (rows of all ranks together); ``N`` = this rank's N shard.  The reference's Triton
    tile hints (``BLOCK_*``, ``stages``) and side streams are accepted for signature parity and have no effect here: tiles
    come from ``gemm_config`` and the gather runs inside the kernel (no streams).

    ``dtype`` int8 / float8_e4m3fn: 8-bit rows plus a fp32 per-row scale workspace; float8_e4m3fn also gets the MXFP8
    scale-chunk workspace used by :func:`ag_gemm_mxfp8` (``K % 128 == 0``)."""
    heap = U.get_heap()
    rank = heap.rank if rank is None else rank
    num_ranks = heap.world if num_ranks is None else num_ranks
    ctx = AllGatherGEMMTensorParallelContext(max_M, N, K, dtype, rank, num_ranks, num_local_ranks or num_ranks,
                                             n_comm_ctas=n_comm_ctas)
    ctx.workspace = heap.tensor((2, max_M, K), dtype)
    if _is_8bit(dtype):
        assert K % 128 == 0, "8-bit ag_gemm needs K % 128 == 0"
        ctx.scale_ws = heap.tensor((2, max_M), torch.float32)
        if dtype != torch.int8:
            ctx.sf_ws = heap.tensor((2, (max_M + 127) // 128, K // 128, 512), torch.uint8)
    ctx.ready = heap.tensor((max(num_ranks, 4),), torch.int32)
    max_ms = (max_M + num_ranks - 1) // num_ranks
    chunks = (max_ms + _CHUNK_ROWS - 1) // _CHUNK_ROWS
    ctx.flags = heap.tensor((2, num_ranks, 256), torch.int32)      # [parity][src][slice], written remotely by the sources
    ctx.phase = torch.zeros(4, dtype=torch.int32, device=heap.device)
    U.barrier_all_host()
    return ctx


def _is_8bit(dtype) -> bool:
    return dtype == torch.int8 or dtype == getattr(torch, "float8_e4m3fn", None)


_WEIGHT_T_CACHE = {}


def _as_nk(B: torch.Tensor) -> torch.Tensor:
    """Return the operand as a K-major ``[N, K]`` matrix.  ``B`` is ``[K, N]``: normally the ``.t()`` view of an
    ``nn.Linear`` weight (free); a genuinely N-major B is transposed once and cached (weights are static)."""
    if B.stride(0) == 1:
        return B.t()
    key = (B.data_ptr(), tuple(B.shape), B._version)
    w = _WEIGHT_T_CACHE.get(key)
    if w is None:
        w = B.t().contiguous()
        _WEIGHT_T_CACHE.clear()
        _WEIGHT_T_CACHE[key] = w
    return w


def default_ag_config(M: int, N: int, K: int, world: int) -> GemmConfig:
    """Tiles of one source rank form one L2 band (``group_m`` = m-tiles per source), so the arrival order of the
    shards is respected while B tiles are re-read once per source rather than once per m-tile."""
    rows = M // max(world, 1)
    nc = (32 if world >= 4 else 16) if world > 1 else 0      # comm CTAs: the push is latency/port bound, 32 SMs fill NVLink at TP>=4
    if rows % 256 == 0 and N >= 256:
        # few tiles (TP8 column shards): 128-wide tiles fill the SMs and halve the tail after the last shard arrives
        bn = 128 if (world > 1 and (M // 256) * ((N + 255) // 256) < 60 and N % 128 == 0) else 256
        return GemmConfig(bn=bn, cta_group=2, group_m=max(1, rows // 256), use_tma_store=True, n_comm_ctas=nc)
    gm = max(1, rows // 128) if rows % 128 == 0 else 1
    if N >= 256:
        return GemmConfig(bn=256, cta_group=1, group_m=gm, use_tma_store=True, n_comm_ctas=nc)
    return GemmConfig(bn=128, cta_group=1, group_m=gm, use_tma_store=True, n_comm_ctas=nc)


def ag_gemm(A: torch.Tensor, B: torch.Tensor, ctx: AllGatherGEMMTensorParallelContext,
            gemm_config: Optional[GemmConfig] = None, straggler_option=None, debug: bool = False,
            out: Optional[torch.Tensor] = None, skip_wait: bool = False, profiler=None, transport: str = "auto",
            all_to_all: bool = False, kslices: int = 0, comm_groups: int = 0, tail_pct: int = 0, scale_a=None,
            scale_b=None) -> torch.Tensor:
    """A: ``[M/W, K]`` local shard, B: ``[K, N/W]`` -> ``[M, N/W]``.  ``skip_wait`` runs the GEMM-only twin
    (flags ignored) used to measure exposed communication, like the reference's ``fake_barrier`` path.

    ``transport="auto"`` (default): ``sm_k`` when ``M/W % 128 == 0``, else ``sm`` (override with env ``TD_AG_TRANSPORT``).
    ``transport="sm_k"``: comm CTAs push the shard K slice by K slice to every peer with unicast stores -- rows are read once,
    one release fence per (CTA, slice) covers all destinations, and every tile follows the arrival of its K slices
    (``kslices``, default 2; ``comm_groups`` groups of CTAs push alternate slices; ``tail_pct`` > 0 makes the LAST round of
    slices carry only that percentage of K, so the MMAs left after the last byte has landed are a few k-blocks).
    ``transport="sm"``: row-sliced P2P push, one fence per (CTA, destination) -- kept for ragged shards and the all-to-all flavour.
    ``transport="copy_engine"``: the
    shard is pushed by the DMA engines on a side stream (one ``cudaMemcpyAsync`` + one release-flag kernel per peer, as
    the reference's copy-engine producer, allgather.py:100-124) while all SMs run GEMM tiles that wait on the same
    per-source flags; not CUDA-graph replayable (flag values are written from the host-tracked phase).
    ``transport="multicast"``: comm CTAs write the shard once to the NVLS multicast alias in ``kslices`` K slices (default 8);
    the ``n_comm_ctas`` CTAs form ``comm_groups`` groups (default 3) that push alternate slices, so that many release fences
    (~7 us of latency each after NVLink stores, measured) are in flight at once.

    ``all_to_all=True``: A is ``[W * Ms, K]`` and row block d goes to rank d (instead of the same shard to everyone);
    the result is ``concat_s(block from rank s) @ B`` -- the AllToAll + GEMM of the Ulysses o-projection
    (reference all_to_all_single_gemm.py:74-188) in the same single kernel.

    8-bit ``A`` (int8 / float8_e4m3fn, context of the same dtype) and ``B`` (``.t()`` view of an 8-bit ``[N/W, K]`` weight): the
    result is bf16 ``(gathered A @ B) * scale_a[row] * scale_b[col]``, as :func:`gemm_scaled`.  ``scale_a``: None, per-tensor (THIS
    rank's scale: every rank quantised its own shard) or per-row ``[M/W]``; ``scale_b``: None, per-tensor or per-channel ``[N/W]``.
    Transports ``sm_k`` / ``multicast`` / ``sm`` (ragged shards on ``sm``); not ``copy_engine`` or ``all_to_all``."""
    if _is_8bit(A.dtype):
        return _ag_gemm_q8(A, B, ctx, gemm_config, straggler_option, out, skip_wait, profiler, transport, all_to_all,
                           kslices, comm_groups, tail_pct, scale_a, scale_b)
    W = ctx.num_ranks
    Ms, K = A.shape
    if all_to_all:
        assert Ms % W == 0
        Ms //= W
    Bnk = _as_nk(B)
    N = Bnk.shape[0]
    M = Ms * W
    assert K == ctx.K and Bnk.shape[1] == K and M <= ctx.max_M and A.dtype == ctx.dtype == Bnk.dtype
    if not A.is_cuda:
        return _ag_gemm_host(A, Bnk, ctx, out, all_to_all)
    if out is None:
        out = torch.empty((M, N), dtype=A.dtype, device=A.device)
    cfg = gemm_config or default_ag_config(M, N, K, W)
    if W == 1:
        from .gemm import gemm
        return gemm(A, Bnk, out=out, config=GemmConfig(cfg.bn, cfg.cta_group, 8, cfg.use_tma_store, cfg.num_sms, 0))
    if straggler_option and straggler_option[0] == ctx.rank:
        torch.cuda._sleep(int(straggler_option[1]))
    heap = U.get_heap()
    A = A.contiguous()
    if transport == "auto":
        transport = resolve_transport(Ms, all_to_all)
    ph = ctx.host_phase + 1
    # zero-copy (A already sits in my slot of the workspace half this call uses) is decided from the HOST mirror of the call
    # counter; inside a CUDA-graph capture the kernel's device-side parity alternates on replay, so it is never assumed there
    zero_copy = ((not all_to_all) and (not torch.cuda.is_current_stream_capturing()) and heap.contains(A)
                 and A.data_ptr() == ctx.workspace[ph & 1][ctx.rank * Ms:].data_ptr())
    assert not (all_to_all and transport == "copy_engine"), "all_to_all flavour uses the in-kernel push"
    args = _C.GemmArgs()
    args.mode = 1
    ws_buf_bytes = ctx.max_M * K * A.element_size()
    fill_common(args, M, ctx.workspace.data_ptr(), K, Bnk, out.data_ptr(), M, out.stride(0), M, N, K, cfg,
                A.dtype == torch.bfloat16)
    args.a_nbuf, args.a_buf_stride_bytes = 2, ws_buf_bytes
    tm = 128 * cfg.cta_group
    args.m_rot = (ctx.rank * Ms) // tm
    r, w, base, stride, mc = U.symm_ctx_fields()
    args.rank, args.world, args.symm_base, args.symm_stride, args.mc_base = r, w, base, stride, mc
    args.phase = ctx.phase.data_ptr()
    args.ag_rows_per_rank, args.ag_copy_local, args.ag_skip_wait = Ms, 2 if all_to_all else (0 if zero_copy else 1), int(skip_wait)
    args.ag_a_local, args.ag_ws, args.ag_ws_buf_bytes = A.data_ptr(), ctx.workspace.data_ptr(), ws_buf_bytes
    args.ag_flags, args.ag_ready = ctx.flags.data_ptr(), ctx.ready.data_ptr()
    if skip_wait:
        args.n_comm_ctas = 0
    if transport == "multicast" and not skip_wait:
        # NVLS: comm CTAs write the shard once to the multicast alias of the workspace (csrc/gemm_sm100.cuh, ag_multicast)
        assert not all_to_all and U.is_nvshmem_multimem_supported() and Ms % 128 == 0
        args.ag_skip_wait = 3
        args.n_comm_ctas = max(2, min(cfg.n_comm_ctas or 24, 64))
        args.ag_kslices = (kslices & 255) | (comm_groups << 8) | ((tail_pct & 255) << 16)
    if transport == "sm_k" and not skip_wait:
        # P2P K-sliced push: rows read once, stored to every peer, ONE release fence per (comm CTA, K slice) for all destinations
        assert not all_to_all and Ms % 128 == 0
        args.ag_skip_wait = 4
        args.n_comm_ctas = max(2, min(cfg.n_comm_ctas or 32, 64))
        args.ag_kslices = (kslices & 255) | (comm_groups << 8) | ((tail_pct & 255) << 16)
    if transport == "copy_engine" and not skip_wait:
        _ce_push(ctx, A, ph, Ms, K)
        args.ag_skip_wait, args.ag_copy_local, args.n_comm_ctas = 2, 1, 0
    if profiler is not None:
        profiler.attach(args)
    _C.check(_C.cuda_lib().td_gemm_launch(C.byref(args), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
             "td_gemm_launch(ag)")
    ctx.host_phase = ph
    if transport == "copy_engine" and not skip_wait:
        torch.cuda.current_stream().wait_stream(ctx._ce_stream)     # A may be reused only after the DMA reads finished
    return out


def _ag_gemm_q8(A, B, ctx, gemm_config, straggler_option, out, skip_wait, profiler, transport, all_to_all, kslices, comm_groups,
                tail_pct, scale_a, scale_b):
    from .gemm import _Q8_CODE, _scale_vec, gemm_scaled
    W = ctx.num_ranks
    Ms, K = A.shape
    Bnk = _as_nk(B)
    N = Bnk.shape[0]
    M = Ms * W
    if all_to_all:
        raise NotImplementedError("ag_gemm: the all-to-all flavour takes 16-bit inputs")
    if A.dtype != ctx.dtype or Bnk.dtype != A.dtype:
        raise ValueError(f"ag_gemm: 8-bit A, B and context must share one dtype (A {A.dtype}, B {Bnk.dtype}, context {ctx.dtype})")
    assert K == ctx.K and Bnk.shape[1] == K and M <= ctx.max_M
    sa = _scale_vec(scale_a, Ms, A.device)        # per-tensor -> MY rows only, before the gather
    sb = _scale_vec(scale_b, N, A.device)
    if transport not in ("auto", "sm_k", "multicast", "sm"):
        raise NotImplementedError(f"ag_gemm: transport {transport!r} takes 16-bit inputs; 8-bit uses sm_k, multicast or sm")
    if not A.is_cuda:
        return _ag_gemm_host(A, Bnk, ctx, out, scale_a=sa, scale_b=sb)
    if out is None:
        out = torch.empty((M, N), dtype=torch.bfloat16, device=A.device)
    cfg = gemm_config or default_ag_config(M, N, K, W)
    if W == 1:
        return gemm_scaled(A, Bnk, sa, sb, out=out, config=GemmConfig(cfg.bn, cfg.cta_group, 8, cfg.use_tma_store, cfg.num_sms, 0))
    if transport == "auto":
        transport = resolve_transport(Ms)
        if transport not in ("sm_k", "multicast", "sm"):
            raise NotImplementedError(f"ag_gemm: transport {transport!r} takes 16-bit inputs; 8-bit uses sm_k, multicast or sm")
    A = A.contiguous()
    args = _q8_args(A, Bnk, ctx, out, cfg, transport, skip_wait, kslices, comm_groups, tail_pct, straggler_option)
    args.is_bf16 = _Q8_CODE[A.dtype]
    if sa is not None:
        args.scale_a, args.ag_scale_ws = sa.data_ptr(), ctx.scale_ws.data_ptr()
    args.scale_b = sb.data_ptr() if sb is not None else None
    return _launch_ag(args, ctx, out, profiler)


def _q8_args(A, Bnk, ctx, out, cfg, transport, skip_wait, kslices, comm_groups, tail_pct, straggler_option):
    """Launch arguments shared by the 8-bit entry points (A already validated: an 8-bit ``[M/W, K]`` shard)."""
    W = ctx.num_ranks
    Ms, K = A.shape
    N, M = Bnk.shape[0], Ms * W
    if transport in ("sm_k", "multicast") and Ms % 128:
        raise ValueError(f"ag_gemm: transport {transport!r} needs (M / world) % 128 == 0")
    if transport == "multicast" and not U.is_nvshmem_multimem_supported():
        raise RuntimeError("ag_gemm: multicast transport needs NVLS multicast")
    if straggler_option and straggler_option[0] == ctx.rank:
        torch.cuda._sleep(int(straggler_option[1]))
    args = _C.GemmArgs()
    args.mode = 1
    ws_buf_bytes = ctx.max_M * K
    fill_common(args, M, ctx.workspace.data_ptr(), K, Bnk, out.data_ptr(), M, out.stride(0), M, N, K, cfg, True)
    args.a_nbuf, args.a_buf_stride_bytes = 2, ws_buf_bytes
    args.m_rot = (ctx.rank * Ms) // (128 * cfg.cta_group)
    r, w, base, stride, mc = U.symm_ctx_fields()
    args.rank, args.world, args.symm_base, args.symm_stride, args.mc_base = r, w, base, stride, mc
    args.phase = ctx.phase.data_ptr()
    # always pushed from the caller's shard (no zero-copy): the scales of my rows come from the caller's tensors too
    args.ag_rows_per_rank, args.ag_copy_local, args.ag_skip_wait = Ms, 1, int(skip_wait)
    args.ag_a_local, args.ag_ws, args.ag_ws_buf_bytes = A.data_ptr(), ctx.workspace.data_ptr(), ws_buf_bytes
    args.ag_flags, args.ag_ready = ctx.flags.data_ptr(), ctx.ready.data_ptr()
    if skip_wait:
        args.n_comm_ctas = 0
    elif transport in ("sm_k", "multicast"):
        mcast = transport == "multicast"
        args.ag_skip_wait = 3 if mcast else 4
        args.n_comm_ctas = max(2, min(cfg.n_comm_ctas or (24 if mcast else 32), 64))
        args.ag_kslices = (kslices & 255) | (comm_groups << 8) | ((tail_pct & 255) << 16)
    return args


def _launch_ag(args, ctx, out, profiler):
    if profiler is not None:
        profiler.attach(args)
    _C.check(_C.cuda_lib().td_gemm_launch(C.byref(args), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
             "td_gemm_launch(ag, 8-bit)")
    ctx.host_phase += 1
    return out


def ag_gemm_mxfp8(a, b, ctx: AllGatherGEMMTensorParallelContext, out: Optional[torch.Tensor] = None,
                  gemm_config: Optional[GemmConfig] = None, transport: str = "auto", kslices: int = 0, comm_groups: int = 0,
                  tail_pct: int = 0, skip_wait: bool = False, straggler_option=None, profiler=None) -> torch.Tensor:
    """Block-scaled fp8 AllGather + GEMM: ``a`` is this rank's :class:`triton_dist.ops.fp8.MXFP8Tensor` shard ``[M/W, K]``,
    ``b`` the MXFP8 weight ``[N/W, K]``; returns bf16 ``[M, N/W]`` = ``dequant(gathered a) @ dequant(b).T``.  The e4m3 rows and
    their UE8M0 scale chunks are gathered together (``M/W % 128 == 0``: one 512-byte chunk covers 128 rows x 128 K); the
    context must have been created with ``dtype=torch.float8_e4m3fn``.  Transports as :func:`ag_gemm` (``sm_k`` / ``multicast``
    / ``sm``).  At world 1 this is :func:`gemm_mxfp8`."""
    from .fp8 import MXFP8Tensor, dequantize_mxfp8, fill_fp8, gemm_mxfp8
    W = ctx.num_ranks
    Ms, K = a.shape
    N = b.shape[0]
    M = Ms * W
    if ctx.sf_ws is None:
        raise ValueError("ag_gemm_mxfp8 needs a context created with dtype=torch.float8_e4m3fn")
    if Ms % 128:
        raise ValueError("ag_gemm_mxfp8 needs (M / world) % 128 == 0 (one scale chunk covers 128 rows)")
    assert K == ctx.K and b.shape[1] == K and M <= ctx.max_M and a.q.dtype == b.q.dtype == torch.float8_e4m3fn
    assert a.q.is_contiguous() and a.sf.is_contiguous(), "ag_gemm_mxfp8: the shard and its scale chunks must be contiguous"
    if transport not in ("auto", "sm_k", "multicast", "sm"):
        raise NotImplementedError(f"ag_gemm_mxfp8: transport {transport!r} is not supported; use sm_k, multicast or sm")
    if not a.q.is_cuda:
        return _ag_gemm_host(a.q, b, ctx, out, sf=a.sf)
    if out is None:
        out = torch.empty((M, N), dtype=torch.bfloat16, device=a.q.device)
    cg = 2 if Ms % 256 == 0 else 1
    cfg = gemm_config or GemmConfig(bn=128, cta_group=cg, group_m=max(1, Ms // (128 * cg)), use_tma_store=True,
                                    n_comm_ctas=32 if W >= 4 else 16)
    if W == 1:
        return gemm_mxfp8(a, b, out=out, config=GemmConfig(cfg.bn, cfg.cta_group, 8, cfg.use_tma_store, cfg.num_sms, 0))
    if transport == "auto":
        transport = resolve_transport(Ms)
        if transport not in ("sm_k", "multicast", "sm"):
            raise NotImplementedError(f"ag_gemm_mxfp8: transport {transport!r} is not supported; use sm_k, multicast or sm")
    args = _q8_args(a.q, b.q, ctx, out, cfg, transport, skip_wait, kslices, comm_groups, tail_pct, straggler_option)
    buf_chunks = ctx.sf_ws.shape[1] * ctx.sf_ws.shape[2]
    fill_fp8(args, MXFP8Tensor(ctx.workspace[0], ctx.sf_ws.view(-1, K // 128, 512), (2 * ctx.max_M, K)), b)
    args.ag_sfa_local, args.ag_sfa_buf_chunks = a.sf.data_ptr(), buf_chunks
    return _launch_ag(args, ctx, out, profiler)


def resolve_transport(rows_per_rank: int, all_to_all: bool = False) -> str:
    """The transport ``transport="auto"`` picks (env ``TD_AG_TRANSPORT`` overrides)."""
    import os
    forced = os.environ.get("TD_AG_TRANSPORT", "")
    if forced:
        return forced
    if (not all_to_all) and rows_per_rank % 128 == 0:
        return "sm_k"
    return "sm"


def _ce_push(ctx, A, ph, Ms, K):
    """Copy-engine transport: push my shard into every rank's workspace[ph & 1] and raise flag[src=me][0] = ph there."""
    from .. import language as dl
    heap = U.get_heap()
    if getattr(ctx, "_ce_stream", None) is None:
        ctx._ce_stream = torch.cuda.Stream(priority=-1)
    W, me, par = ctx.num_ranks, ctx.rank, ph & 1
    ctx._ce_stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(ctx._ce_stream):
        for dist_ in range(W):
            d = (me - dist_ + W) % W
            dst = heap.peer_view(ctx.workspace, d)[par, me * Ms:(me + 1) * Ms, :K]
            dst.copy_(A, non_blocking=True)
            dl.notify(ctx.flags[par, me, 0:1], d, signal=ph, sig_op="set")


def gemm_only(A_full: torch.Tensor, B: torch.Tensor, out: Optional[torch.Tensor] = None,
              gemm_config: Optional[GemmConfig] = None) -> torch.Tensor:
    """The local GEMM on already-gathered rows (what the fused kernel must hide the all-gather behind)."""
    from .gemm import gemm
    return gemm(A_full, _as_nk(B), out=out, config=gemm_config)


# reference names (allgather_gemm.py:725-800)
def gemm_persistent(A, B, out=None, **_):
    return gemm_only(A, B, out)


gemm_non_persistent = gemm_persistent


# ------------------------------------------------------------------------------------------------------------
# emulation (no GPU): same protocol on the shared-memory heap
# ------------------------------------------------------------------------------------------------------------
def _ag_gemm_host(A, Bnk, ctx, out, all_to_all=False, scale_a=None, scale_b=None, sf=None):
    """Same push protocol as the device kernel: my shard goes into EVERY rank's workspace (nearest consumer first),
    each arrival is published with a release flag carrying the phase number; the GEMM consumes sources in arrival
    order after acquiring their flags.  Workspaces are double buffered by call parity, nothing is reset.

    8-bit shards travel as 8-bit rows together with their per-row scales (``scale_a``, fp32 [Ms]) or MXFP8 scale chunks
    (``sf``, [Ms / 128, K / 128, 512]) under the same flag, and are dequantised by the consumer after the flag wait.
    ``Bnk`` is then an 8-bit ``[N, K]`` weight with ``scale_b`` ([N] or None), or an MXFP8Tensor."""
    import ctypes
    heap = U.get_heap()
    lib = _C.host_lib()
    W, me = ctx.num_ranks, ctx.rank
    Ms, K = A.shape
    if all_to_all:
        Ms //= W
    ctx.host_phase += 1
    ph = ctx.host_phase
    par = ph & 1
    timeout = U.get_int_env("TD_HOST_TIMEOUT_US", 60_000_000)
    flag_off = lambda src: ctx.flags[par, src, 0:1].data_ptr()
    # 1. push (producer role)
    for dist_ in range(W):
        d = (me - dist_ + W) % W
        dst_ws = heap.peer_view(ctx.workspace, d)[par]
        dst_ws[me * Ms:(me + 1) * Ms].copy_(A[d * Ms:(d + 1) * Ms] if all_to_all else A)
        if scale_a is not None:
            heap.peer_view(ctx.scale_ws, d)[par, me * Ms:(me + 1) * Ms].copy_(scale_a)
        if sf is not None:
            heap.peer_view(ctx.sf_ws, d)[par, me * Ms // 128:(me + 1) * Ms // 128].copy_(sf)
        lib.tdh_notify32(ctypes.c_void_p(heap.peer_ptr(flag_off(me), d)), ph, 1)
    # 2. consume in arrival order
    quant = _is_8bit(A.dtype)
    out_dtype = torch.bfloat16 if quant else A.dtype
    if sf is not None:
        from .fp8 import MXFP8Tensor, dequantize_mxfp8
        bt = dequantize_mxfp8(Bnk).t()
    else:
        bt = Bnk.float().t()
    N = bt.shape[1]
    if out is None:
        out = torch.empty((Ms * W, N), dtype=out_dtype)
    ws = ctx.workspace[par]
    for j in range(W):
        s = (me + j) % W
        if lib.tdh_wait32(ctypes.c_void_p(flag_off(s)), ph, 1, timeout):
            raise TimeoutError(f"ag_gemm: shard of rank {s} never arrived (phase {ph})")
        rows = ws[s * Ms:(s + 1) * Ms]
        if sf is not None:
            a = dequantize_mxfp8(MXFP8Tensor(rows, ctx.sf_ws[par, s * Ms // 128:(s + 1) * Ms // 128], (Ms, ctx.K)))
        else:
            a = rows.float()
        acc = a @ bt
        if scale_a is not None or scale_b is not None:     # the kernel's order: acc * (scale_a[row] * scale_b[col])
            sa = ctx.scale_ws[par, s * Ms:(s + 1) * Ms, None] if scale_a is not None else torch.ones(Ms, 1)
            acc = acc * (sa * (scale_b[None, :] if scale_b is not None else 1.0))
        out[s * Ms:(s + 1) * Ms] = acc.to(out_dtype)
    return out


# ------------------------------------------------------------------------------------------------------------
# autotuned entry point (reference: ag_gemm is wrapped by triton_dist.tune.autotune, allgather_gemm.py:565-619)
# ------------------------------------------------------------------------------------------------------------
from ..tune import autotune  # noqa: E402

AG_GEMM_TUNE_SPACE = (
    [dict(transport="sm_k", bn=bn, cta_group=cg, n_comm=nc, kslices=ks, groups=gr, tail=tail)
     for (bn, cg) in ((256, 2), (128, 2), (256, 1)) for (nc, ks, gr, tail) in ((32, 2, 1, 0), (32, 4, 2, 12), (48, 6, 2, 10), (32, 1, 1, 0))]
    + [dict(transport="multicast", bn=128, cta_group=2, n_comm=24, kslices=8, groups=3, tail=0),
       dict(transport="sm", bn=256, cta_group=2, n_comm=16, kslices=0, groups=0, tail=0),
       dict(transport="sm", bn=128, cta_group=2, n_comm=32, kslices=0, groups=0, tail=0)])


def ag_gemm_config_space():
    """The search space of ``ag_gemm_tuned`` (reference: allgather_gemm.py ``ag_gemm_config_space``)."""
    return list(AG_GEMM_TUNE_SPACE)


def ag_gemm_key_fn(A, B, ctx, **_):
    return f"{tuple(A.shape)}x{tuple(B.shape)}@tp{ctx.num_ranks}"


def _ag_prune(cfg, A, B, ctx, **_):
    Ms = A.shape[0]
    if cfg["transport"] in ("sm_k", "multicast") and Ms % 128:
        return False
    if cfg["transport"] == "multicast" and not U.is_nvshmem_multimem_supported():
        return False
    return cfg["cta_group"] == 1 or Ms % 256 == 0


@autotune(AG_GEMM_TUNE_SPACE, key_fn=ag_gemm_key_fn, prune_fn=_ag_prune,
          warmup=3, rep=8)
def ag_gemm_tuned(A: torch.Tensor, B: torch.Tensor, ctx: AllGatherGEMMTensorParallelContext, out: Optional[torch.Tensor] = None,
                  config: Optional[dict] = None) -> torch.Tensor:
    """``ag_gemm`` with transport / tile / comm-CTA configuration chosen by the function-level autotuner: every candidate is
    timed with CUDA events, the MAX over ranks decides (pass ``autotune_pg=group``), the winner is cached on disk per
    (shape, world size, GPU).  ``ag_gemm_tuned(A, B, ctx, autotune=False)`` uses the first (default) configuration.
    16-bit inputs only: call :func:`ag_gemm` with ``scale_a`` / ``scale_b`` for 8-bit ones."""
    if _is_8bit(A.dtype):
        raise NotImplementedError("ag_gemm_tuned takes 16-bit inputs; use ag_gemm(..., scale_a=, scale_b=) for 8-bit ones")
    c = config or AG_GEMM_TUNE_SPACE[0]
    Ms = A.shape[0]
    cfg = GemmConfig(c["bn"], c["cta_group"], max(1, Ms // (128 * c["cta_group"])), True, 0, c["n_comm"])
    return ag_gemm(A, B, ctx, gemm_config=cfg, out=out, transport=c["transport"] if A.is_cuda else "auto", kslices=c["kslices"],
                   comm_groups=c["groups"], tail_pct=c["tail"])


ag_gemm_prune_fn = _ag_prune
