#!/usr/bin/env python
"""8-bit AllGather + GEMM vs bf16 on B200s (run under torchrun, one process per GPU; there is no CPU fallback).

    python -m torch.distributed.run --nproc-per-node 8 scripts/bench_ag_gemm_q8.py --out profiles/ag_gemm_q8_8xB200.json

Times, on the device with CUDA events, inside ONE interleaved loop (every variant runs once per round, max over ranks per call):
  bf16 ag_gemm; int8 and e4m3 ag_gemm with per-row scale_a and per-channel scale_b; ag_gemm_mxfp8; every variant's GEMM-only twin
  (skip_wait: same kernel, no waits => exposed communication = fused - twin); the non-fused 8-bit baseline = NCCL all-gather of the
  8-bit rows + their scales, then gemm_scaled / gemm_mxfp8.
Inputs rotate through enough sets that a round's working set exceeds the 126 MB L2.  Roofline of a variant = max(bytes that
cross NVLink into one GPU / 770 GB/s, FLOPs / peak), peak from the data sheet (dense, per GPU: 2250 TFLOP/s bf16, 4500 fp8 / int8).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"baseline_ag": (4096, 4096, 4096), "qwen3_32b_gate_up": (8192, 2 * 25600, 5120)}
NVLINK_GBPS = 770.0
PEAK_TFLOPS = {"bf16": 2250.0, "8bit": 4500.0}      # data sheet, dense, per GPU (not measured here)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        sys.exit("bench_ag_gemm_q8: needs a GPU (no CPU fallback)")
    import triton_dist.utils as U
    from triton_dist.ops.ag_gemm import ag_gemm, ag_gemm_mxfp8, create_ag_gemm_context
    from triton_dist.ops.fp8 import MXFP8Tensor, gemm_mxfp8, quantize_mxfp8
    from triton_dist.ops.gemm import gemm_scaled
    U.initialize_distributed(seed=0)
    W, me, grp, dev = U.world_size(), U.rank(), U.get_triton_dist_world(), torch.device("cuda")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    result = dict(world=W, gpu=smi[torch.cuda.current_device()] if smi else "unknown", nvlink_gbps_assumed=NVLINK_GBPS,
                  peak_tflops_data_sheet=PEAK_TFLOPS, rounds=args.rounds, shapes={})
    for name, (M, N, K) in SHAPES.items():
        Ms, Nr = M // W, N // W
        nset = max(2, int(2 * 126e6 // (Ms * K * 2 + Nr * K * 2)) + 1)
        ctxs = {dt: create_ag_gemm_context(M, Nr, K, dt) for dt in (torch.bfloat16, torch.int8, torch.float8_e4m3fn)}
        sets = []
        for _ in range(nset):
            x = torch.randn(Ms, K, device=dev, dtype=torch.bfloat16)
            w = torch.randn(Nr, K, device=dev, dtype=torch.bfloat16) * K ** -0.5
            sx, sw = x.abs().amax(1).float() / 127, w.abs().amax(1).float() / 127
            sets.append(dict(x=x, w=w, xi=(x / sx[:, None]).round().to(torch.int8), wi=(w / sw[:, None]).round().to(torch.int8),
                             sxi=sx, swi=sw, x8=(x / (sx[:, None] * 127 / 448)).to(torch.float8_e4m3fn),
                             w8=(w / (sw[:, None] * 127 / 448)).to(torch.float8_e4m3fn), sx8=sx * 127 / 448, sw8=sw * 127 / 448,
                             xm=quantize_mxfp8(x), wm=quantize_mxfp8(w)))
        full8 = torch.empty(M, K, device=dev, dtype=torch.uint8)
        fulls = torch.empty(M, device=dev, dtype=torch.float32)
        fullsf = torch.empty((M // 128) * (K // 128) * 512, device=dev, dtype=torch.uint8)

        def nccl_q8(s, q, sa, sb):
            dist.all_gather_into_tensor(full8, s[q].view(torch.uint8), group=grp)
            dist.all_gather_into_tensor(fulls, s[sa], group=grp)
            return gemm_scaled(full8.view(s[q].dtype), s[q.replace("x", "w")], fulls, s[sb])

        def nccl_mx(s):
            dist.all_gather_into_tensor(full8, s["xm"].q.view(torch.uint8), group=grp)
            dist.all_gather_into_tensor(fullsf, s["xm"].sf.view(-1), group=grp)
            return gemm_mxfp8(MXFP8Tensor(full8.view(torch.float8_e4m3fn), fullsf.view(M // 128, K // 128, 512), (M, K)), s["wm"])

        bf, i8, f8 = ctxs[torch.bfloat16], ctxs[torch.int8], ctxs[torch.float8_e4m3fn]
        variants = {
            "bf16": lambda s: ag_gemm(s["x"], s["w"].t(), bf),
            "bf16_twin": lambda s: ag_gemm(s["x"], s["w"].t(), bf, skip_wait=True),
            "int8": lambda s: ag_gemm(s["xi"], s["wi"].t(), i8, scale_a=s["sxi"], scale_b=s["swi"]),
            "int8_twin": lambda s: ag_gemm(s["xi"], s["wi"].t(), i8, scale_a=s["sxi"], scale_b=s["swi"], skip_wait=True),
            "e4m3": lambda s: ag_gemm(s["x8"], s["w8"].t(), f8, scale_a=s["sx8"], scale_b=s["sw8"]),
            "e4m3_twin": lambda s: ag_gemm(s["x8"], s["w8"].t(), f8, scale_a=s["sx8"], scale_b=s["sw8"], skip_wait=True),
            "mxfp8": lambda s: ag_gemm_mxfp8(s["xm"], s["wm"], f8),
            "mxfp8_twin": lambda s: ag_gemm_mxfp8(s["xm"], s["wm"], f8, skip_wait=True),
        }
        if W > 1:
            variants["nccl_int8"] = lambda s: nccl_q8(s, "xi", "sxi", "swi")
            variants["nccl_e4m3"] = lambda s: nccl_q8(s, "x8", "sx8", "sw8")
            variants["nccl_mxfp8"] = nccl_mx
        times = {k: [] for k in variants}
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in variants]
        for r in range(args.warmup + args.rounds):
            s = sets[r % nset]
            for (k, fn), (e0, e1) in zip(variants.items(), ev):
                U.barrier_all_on_stream()
                e0.record()
                fn(s)
                e1.record()
            torch.cuda.synchronize()
            if r >= args.warmup:
                for k, (e0, e1) in zip(variants, ev):
                    times[k].append(e0.elapsed_time(e1) * 1e3)
        t = torch.tensor([times[k] for k in variants], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=grp)          # per call: the slowest rank
        med = {k: float(t[i].median()) for i, k in enumerate(variants)}
        spread = {k: [float(t[i].min()), float(t[i].max())] for i, k in enumerate(variants)}
        flops = 2.0 * M * Nr * K
        roof = {}
        for k in ("bf16", "int8", "e4m3", "mxfp8"):
            esz = 2 if k == "bf16" else 1
            sbytes = (M - Ms) * ((4 if k in ("int8", "e4m3") else 0) + (K // 32 if k == "mxfp8" else 0))
            nv_us = ((M - Ms) * K * esz + sbytes) / (NVLINK_GBPS * 1e3)
            mma_us = flops / (PEAK_TFLOPS["bf16" if k == "bf16" else "8bit"] * 1e6)
            roof[k] = dict(nvlink_us=nv_us, mma_us_data_sheet=mma_us, roofline_us=max(nv_us, mma_us),
                           fraction_of_roofline=max(nv_us, mma_us) / med[k], exposed_comm_us=med[k] - med[k + "_twin"])
        result["shapes"][name] = dict(M=M, N_per_rank=Nr, K=K, input_sets=nset, median_us=med, min_max_us=spread, roofline=roof,
                                      speedup_vs_bf16={k: med["bf16"] / med[k] for k in ("int8", "e4m3", "mxfp8")},
                                      speedup_vs_nccl=({k: med["nccl_" + k] / med[k] for k in ("int8", "e4m3", "mxfp8")}
                                                       if W > 1 else "not measured (world 1)"))
        U.barrier_all_host()
        for c in ctxs.values():
            c.finalize()
        del sets
        torch.cuda.empty_cache()
    if me == 0:
        print(json.dumps(result))
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(result, f, indent=1)
    U.finalize_distributed()


if __name__ == "__main__":
    main()
