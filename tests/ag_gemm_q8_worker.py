"""Multi-process worker of the 8-bit AllGather + GEMM tests (tests/test_ag_gemm_q8_{cpu,gpu}.py), launched by torchrun on CPU
(gloo + the shared-memory emulation backend) or on GPUs.  Same pattern as tests/dist_worker.py: fresh random inputs every call,
poisoned workspaces, golden = torch.distributed collective + fp32 matmul on the dequantised operands, stragglers.
Usage: torchrun ... tests/ag_gemm_q8_worker.py <case> [<case> ...]
"""
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import triton_dist.utils as U  # noqa: E402


def run_cases(cases, nproc, timeout=900, env_extra=None):
    """Run the named cases of this worker under torchrun (127.0.0.1 rendezvous); raise with the output on failure."""
    from _launch import free_port
    env = dict(os.environ)
    env.setdefault("OMP_NUM_THREADS", "2")
    env.update(env_extra or {})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), os.path.abspath(__file__)] + list(cases)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
    if r.returncode != 0:
        raise AssertionError(f"8-bit ag_gemm worker failed (rc={r.returncode})\n--- stdout ---\n{r.stdout[-6000:]}\n"
                             f"--- stderr ---\n{r.stderr[-6000:]}")
    for c in cases:
        assert f"CASE {c} OK" in r.stdout, r.stdout[-3000:]
    return r.stdout


def _assert_close(a, b, atol, rtol, what):
    a, b = a.float().cpu(), b.float().cpu()
    if not torch.allclose(a, b, atol=atol, rtol=rtol):
        err = (a - b).abs()
        raise AssertionError(f"[rank {U.rank()}] {what}: max abs err {err.max().item():.4g} at {err.argmax().item()} "
                             f"(ref max {b.abs().max().item():.4g})")


def _q8_gather(x):
    """dist.all_gather_into_tensor of an 8-bit / fp32 shard (8-bit bytes travel as uint8)."""
    raw = x.view(torch.uint8) if x.dtype != torch.float32 else x
    full = torch.empty((U.world_size() * raw.shape[0],) + tuple(raw.shape[1:]), dtype=raw.dtype, device=raw.device)
    dist.all_gather_into_tensor(full, raw.contiguous(), group=U.get_triton_dist_world())
    return full.view(x.dtype) if x.dtype != torch.float32 else full


def _q8_operands(kind, M, N, K, dev):
    if kind == "int8":
        return (torch.randint(-127, 128, (M, K), device=dev, dtype=torch.int8),
                torch.randint(-127, 128, (N, K), device=dev, dtype=torch.int8))
    return ((torch.randn(M, K, device=dev) * 2).to(torch.float8_e4m3fn), (torch.randn(N, K, device=dev) * 2).to(torch.float8_e4m3fn))


def _q8_check(C, ref, kind, what):
    # int8: the int32 accumulation is exact and the golden multiplies by the scales in the kernel's order, so the only error is
    # the bf16 rounding of the output (relative 2^-8).  e4m3 / MXFP8: the dequantised operands are exact in both, only the order
    # (and width) of the fp32 tensor-core accumulation differs: 0.5 % of the largest output + 1 %.  A scale or a row that lands
    # on the wrong rows moves outputs by tens of percent (scales differ up to 20x between rows and ranks), far outside this.
    if kind == "int8":
        _assert_close(C, ref, 1e-6 * ref.abs().max().item(), 2.0 ** -8, what)
    else:
        _assert_close(C, ref, 5e-3 * ref.abs().max().item(), 1e-2, what)


def _ag_q8_poison(ctx):
    if ctx.workspace.is_cuda:
        ctx.workspace.view(torch.uint8).fill_(0x7F)          # e4m3 NaN bytes (int8: 127 everywhere)
        ctx.scale_ws.fill_(float("nan"))
        if ctx.sf_ws is not None:
            ctx.sf_ws.fill_(0xFF)                             # UE8M0 NaN


def case_ag_gemm_q8():
    """8-bit AllGather + GEMM: int8 / e4m3 shards with per-row or per-tensor scale_a (a different per-tensor scale on every rank) and
    per-channel / per-tensor scale_b, and MXFP8 shards, over every in-kernel transport, vs fp32 math on the dequantised operands
    gathered with all_gather_into_tensor.  Poisoned workspaces, stragglers, fresh inputs every call."""
    from triton_dist.ops.ag_gemm import ag_gemm, ag_gemm_mxfp8, create_ag_gemm_context
    from triton_dist.ops.fp8 import dequantize_mxfp8, quantize_mxfp8
    from triton_dist.ops.gemm import GemmConfig
    dev = U.current_device()
    W, me = U.world_size(), U.rank()
    big = dev.type == "cuda"
    if big:
        # (M, N, K, tile config): 2-CTA and 1-CTA tiles, bn 128 and 256; the last shape has ragged shards (M / W % 128 != 0)
        shapes = [(256 * W, 512, 1024, GemmConfig(256, 2, 1, True, 0, 16)), (256 * W, 384, 512, GemmConfig(128, 2, 1, True, 0, 16)),
                  (128 * W, 256, 768, GemmConfig(128, 1, 1, True, 0, 8)), (128 * W, 512, 512, GemmConfig(256, 1, 1, False, 0, 16)),
                  (100 * W, 256, 384, GemmConfig(128, 1, 1, True, 0, 16))]
        transports = ["sm_k", "sm"] + (["multicast"] if (W > 1 and U.is_nvshmem_multimem_supported()) else [])
    else:
        shapes = [(128 * W, 64, 256, None), (40 * W, 48, 128, None)]
        transports = ["auto"]
    for (M, N, K, cfg) in shapes:
        Ms = M // W
        for kind in ("int8", "e4m3", "mxfp8"):
            if kind == "mxfp8" and Ms % 128:
                continue
            dt = torch.int8 if kind == "int8" else torch.float8_e4m3fn
            ctx = create_ag_gemm_context(M, N, K, dt)
            _ag_q8_poison(ctx)
            for tr in transports:
                if tr in ("sm_k", "multicast") and Ms % 128:
                    continue
                for it in range(4 if big else 3):
                    straggler = (it % W, 2_000_000) if (big and W > 1 and it in (1, 3)) else None
                    ks, gr, tail = ((0, 0, 0), (4, 2, 10), (16, 4, 25), (3, 1, 0))[it]
                    what = f"ag_gemm {kind} [{tr}] {M}x{N}x{K} cfg={cfg} it{it}"
                    if kind == "mxfp8":
                        a = quantize_mxfp8((torch.randn(Ms, K, device=dev) * (1 + me)).to(torch.bfloat16))
                        b = quantize_mxfp8(torch.randn(N, K, device=dev).to(torch.bfloat16))
                        C = ag_gemm_mxfp8(a, b, ctx, gemm_config=cfg, transport=tr, kslices=ks, comm_groups=gr, tail_pct=tail,
                                          straggler_option=straggler)
                        ref = _q8_gather(dequantize_mxfp8(a)) @ dequantize_mxfp8(b).t()
                    else:
                        a, b = _q8_operands(kind, Ms, N, K, dev)
                        per_row, per_chan = it % 2 == 0, it % 3 != 1
                        sa = (torch.rand(Ms, device=dev) * 0.02 + 0.001) if per_row else 0.003 * (1 + me)   # per-tensor: THIS rank's
                        sb = (torch.rand(N, device=dev) * 0.02 + 0.001) if per_chan else torch.tensor(0.0125, device=dev)
                        C = ag_gemm(a, b.t(), ctx, gemm_config=cfg, transport=tr, kslices=ks, comm_groups=gr, tail_pct=tail,
                                    straggler_option=straggler, scale_a=sa, scale_b=sb)
                        sa_full = _q8_gather(sa if per_row else torch.full((Ms,), sa, device=dev))
                        sb_vec = sb if per_chan else sb.expand(N)
                        ref = (_q8_gather(a).float() @ b.float().t()) * (sa_full[:, None] * sb_vec[None, :])
                    assert C.dtype == torch.bfloat16 and C.shape == (M, N), (C.dtype, C.shape)
                    _q8_check(C, ref, "int8" if kind == "int8" else "fp8", what)
            U.barrier_all_host()
            ctx.finalize()


def case_ag_gemm_q8_graph():
    """A captured CUDA graph of the 8-bit AllGather + GEMM, replayed with new inputs: the scale workspaces follow the device-side
    call parity (a replay must not read the scales of the other half)."""
    from triton_dist.ops.ag_gemm import ag_gemm, ag_gemm_mxfp8, create_ag_gemm_context
    from triton_dist.ops.fp8 import dequantize_mxfp8, quantize_mxfp8
    dev = U.current_device()
    if dev.type != "cuda":
        return
    W, me = U.world_size(), U.rank()
    M, N, K = 256 * W, 512, 512
    Ms = M // W
    for kind in ("int8", "e4m3", "mxfp8"):
        for tr in ("sm_k", "sm"):
            ctx = create_ag_gemm_context(M, N, K, torch.int8 if kind == "int8" else torch.float8_e4m3fn)
            _ag_q8_poison(ctx)
            if kind == "mxfp8":
                a = quantize_mxfp8(torch.randn(Ms, K, device=dev).to(torch.bfloat16))
                b = quantize_mxfp8(torch.randn(N, K, device=dev).to(torch.bfloat16))
                run = lambda: ag_gemm_mxfp8(a, b, ctx, transport=tr)
            else:
                a, b = _q8_operands(kind, Ms, N, K, dev)
                sa = torch.rand(Ms, device=dev) * 0.02 + 0.001
                sb = torch.rand(N, device=dev) * 0.02 + 0.001
                run = lambda: ag_gemm(a, b.t(), ctx, transport=tr, scale_a=sa, scale_b=sb)
            run()
            torch.cuda.synchronize()
            U.barrier_all_host()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                C = run()
            for rep in range(4):
                if kind == "mxfp8":
                    n = quantize_mxfp8((torch.randn(Ms, K, device=dev) * (1 + rep + me)).to(torch.bfloat16))
                    a.q.copy_(n.q); a.sf.copy_(n.sf)
                    ref = _q8_gather(dequantize_mxfp8(a)) @ dequantize_mxfp8(b).t()
                else:
                    na, _ = _q8_operands(kind, Ms, N, K, dev)
                    a.copy_(na)
                    sa.copy_(torch.rand(Ms, device=dev) * 0.02 * (1 + rep) + 0.001)
                    ref = (_q8_gather(a).float() @ b.float().t()) * (_q8_gather(sa)[:, None] * sb[None, :])
                torch.cuda.synchronize()
                U.barrier_all_host()
                g.replay()
                torch.cuda.synchronize()
                _q8_check(C, ref, "int8" if kind == "int8" else "fp8", f"graph ag_gemm {kind} [{tr}] replay {rep}")
            U.barrier_all_host()
            del g
            ctx.finalize()


def case_ag_gemm_q8_reject():
    """Combinations outside the 8-bit AllGather + GEMM raise a clear error instead of computing something else."""
    from triton_dist.ops.ag_gemm import ag_gemm, ag_gemm_mxfp8, ag_gemm_tuned, create_ag_gemm_context
    from triton_dist.ops.fp8 import quantize_mxfp8
    dev = U.current_device()
    W = U.world_size()
    M, N, K = 64 * W, 32, 128
    ctx = create_ag_gemm_context(M, N, K, torch.int8)
    a = torch.zeros(M // W, K, dtype=torch.int8, device=dev)
    b = torch.zeros(N, K, dtype=torch.int8, device=dev)

    def expect(exc, fn, what):
        try:
            fn()
        except exc:
            return
        raise AssertionError(f"{what}: no {exc.__name__}")
    expect(NotImplementedError, lambda: ctx.local_input_buffer(M // W), "local_input_buffer on an 8-bit context")
    expect(NotImplementedError, lambda: ag_gemm_tuned(a, b.t(), ctx, autotune=False), "ag_gemm_tuned with 8-bit inputs")
    expect(NotImplementedError, lambda: ag_gemm(a, b.t(), ctx, transport="copy_engine"), "copy_engine with 8-bit inputs")
    expect(NotImplementedError, lambda: ag_gemm(a.repeat(W, 1), b.t(), ctx, all_to_all=True), "all-to-all with 8-bit inputs")
    expect(ValueError, lambda: ag_gemm(a.to(torch.float8_e4m3fn), b.to(torch.float8_e4m3fn).t(), ctx), "e4m3 A on an int8 context")
    expect(ValueError, lambda: ag_gemm_mxfp8(quantize_mxfp8(torch.zeros(M // W, K, device=dev)),
                                             quantize_mxfp8(torch.zeros(N, K, device=dev)), ctx), "MXFP8 on an int8 context")
    U.barrier_all_host()
    ctx.finalize()
    ctx = create_ag_gemm_context(M, N, K, torch.float8_e4m3fn)
    if W > 1:   # 64 rows per rank: one scale chunk covers 128 rows
        expect(ValueError, lambda: ag_gemm_mxfp8(quantize_mxfp8(torch.zeros(M // W, K, device=dev)),
                                                 quantize_mxfp8(torch.zeros(N, K, device=dev)), ctx), "MXFP8 with M / W % 128 != 0")
    U.barrier_all_host()
    ctx.finalize()


def case_tp_mlp_mxfp8():
    """MXFP8 TP MLP forward (quantise -> ag_gemm_mxfp8 -> silu_mul -> quantise -> gemm_rs_mxfp8) vs a golden that applies the same
    quantiser to the same operands: fp32 math on the dequantised values, all-gather / reduce-scatter by torch.distributed."""
    from triton_dist.ops.elementwise import silu_mul
    from triton_dist.ops.fp8 import dequantize_mxfp8, quantize_mxfp8
    from triton_dist.parallel.tp_mlp import TP_MLP
    dev = U.current_device()
    W, me = U.world_size(), U.rank()
    big = dev.type == "cuda"
    H, I, Ms = (1024, 512 * W, 256) if big else (256, 128 * W, 128)
    M = Ms * W
    mlp = TP_MLP(me, W, U.get_triton_dist_world())
    gate_up = (torch.randn(2 * I // W, H, device=dev) * H ** -0.5).to(torch.bfloat16)
    down = (torch.randn(H, I // W, device=dev) * (I ** -0.5)).to(torch.bfloat16)
    mlp._init_parameters_from_shards(gate_up, down)
    mlp._init_ctx(M, mxfp8=True)
    for it in range(3):
        x = torch.randn(Ms, H, device=dev).to(torch.bfloat16)
        out = mlp.dist_triton_mxfp8_fwd(x)
        h = (_q8_gather(dequantize_mxfp8(quantize_mxfp8(x))) @ dequantize_mxfp8(mlp.gate_up_mx).t()).to(torch.bfloat16)
        act = silu_mul(h)
        part = dequantize_mxfp8(quantize_mxfp8(act)) @ dequantize_mxfp8(mlp.down_mx).t()
        if big:
            ref = torch.empty(Ms, H, device=dev)
            dist.reduce_scatter_tensor(ref, part, group=U.get_triton_dist_world())
        else:
            dist.all_reduce(part, group=U.get_triton_dist_world())
            ref = part[me * Ms:(me + 1) * Ms]
        # the golden's h differs from the kernel's in the accumulation order, which can move an activation across an e4m3 rounding
        # boundary (3 mantissa bits) before the down projection; those rare flips average out over I
        _assert_close(out, ref, 3e-2 * ref.abs().max().item(), 5e-2, f"tp_mlp mxfp8 it{it}")
    U.barrier_all_host()
    mlp.finalize()


CASES = {k[5:]: v for k, v in list(globals().items()) if k.startswith("case_")}

if __name__ == "__main__":
    names = sys.argv[1:]
    U.initialize_distributed(seed=1 + int(os.environ.get("RANK", 0)))
    t0 = time.time()
    for name in names:
        CASES[name]()
        U.barrier_all_host()
        U.dist_print(f"CASE {name} OK ({time.time() - t0:.1f}s)", allowed_ranks=[0])
    U.finalize_distributed()
