"""DSL kernels (triton_dist.lk) on a B200: SIMT examples, the tcgen05 GEMM ladder (1-CTA and cta_group::2; run in a subprocess so that
a faulting generated kernel cannot poison the CUDA context of the rest of the suite) and the symmetric-heap kernels on 2 GPUs.
Hardware record: profiles/r2/lk_dsl_gpu_1xB200.log."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_lk_simt_kernels():
    from triton_dist.lk.kernels import simt as K
    torch.manual_seed(0)
    n = 100_003
    x, y = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    ref = 1.5 * x + y
    K.saxpy[(n + 127) // 128](x, y, 1.5, n)
    torch.testing.assert_close(y, ref)

    xb = torch.randn(1 << 20, device="cuda").bfloat16()
    out = torch.zeros(1, device="cuda")
    K.block_sum[148](xb, out, xb.numel())
    torch.testing.assert_close(out[0], xb.float().sum(), atol=0.5, rtol=1e-3)

    m = torch.randn(64, 5000, device="cuda")
    sm = torch.empty_like(m)
    K.softmax_rows[64](m, sm, 5000)
    torch.testing.assert_close(sm, m.softmax(-1), atol=1e-6, rtol=1e-4)

    ids = torch.randint(0, 256, (1 << 18,), device="cuda", dtype=torch.int32)
    cnt = torch.zeros(256, device="cuda", dtype=torch.int32)
    K.histogram[64](ids, cnt, ids.numel(), 256)
    assert torch.equal(cnt, torch.bincount(ids.long(), minlength=256).int())
    attrs = K.softmax_rows.attributes()
    assert attrs["local_bytes"] == 0 and attrs["regs"] > 0


_GEMM_SNIPPET = r"""
import sys, torch
sys.path.insert(0, {root!r})
from triton_dist.lk.kernels.gemm_sm100 import run_gemm
torch.manual_seed(0)
for (M, N, K) in ((256, 256, 128), (512, 768, 512), (1000, 392, 320), (4096, 4096, 4096)):
    a = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
    b = (torch.randn(N, K, device="cuda") * 0.5).bfloat16()
    ref = a.float() @ b.float().t()
    c = run_gemm(a, b, cta_group={cg})
    torch.cuda.synchronize()
    torch.testing.assert_close(c.float(), ref, atol=0.5, rtol=2e-2)
print("LK_GEMM_OK")
"""


@pytest.mark.parametrize("cg", [1, 2])
def test_lk_gemm_ladder(cg):
    r = subprocess.run([sys.executable, "-c", _GEMM_SNIPPET.format(root=ROOT, cg=cg)], capture_output=True, text=True, timeout=150, cwd=ROOT)
    assert r.returncode == 0 and "LK_GEMM_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_lk_symmetric_heap_kernels_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["lk"], nproc=2, timeout=240)


def test_shmem_header_two_gpus():
    """csrc/td/shmem.cuh (NVSHMEM-style device API) through a JIT kernel + the stream-ordered Python mirror."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["shmem"], nproc=2, timeout=240)


def test_allgather_multimem_two_gpus():
    """NVLS all-gather kernels (multimem push, multimem LL) written after the GPU budget of the round was spent."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["allgather_mc"], nproc=2, timeout=240)


def test_gemm_a2a_quantised_two_gpus():
    """int8 GEMM + all-to-all: the two-kernel path (validated halves) and the fused one-kernel variant (new combination)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["gemm_a2a_q8"], nproc=2, timeout=240)


def test_sp_varlen_two_gpus():
    """Packed variable-length context-parallel attention (one KV gather for the batch, tcgen05 flash per sequence)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["sp_varlen"], nproc=2, timeout=240)


def _isolated(code: str, marker: str, timeout: int = 150):
    """Run a snippet in its own process: a faulting or hanging kernel cannot take the rest of the suite with it."""
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r)\n" % ROOT + code], capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0 and marker in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


_VARLEN_SNIPPET = r"""
import torch
from triton_dist.ops.flash_attn import flash_attn_reference, flash_attn_varlen
causal = {causal}
torch.manual_seed(3)
lens_q, lens_k = [5, 130, 64, 512, 1], [9, 130, 200, 512, 77]
cq = torch.tensor([0] + list(torch.tensor(lens_q).cumsum(0)), dtype=torch.int32, device="cuda")
ck = torch.tensor([0] + list(torch.tensor(lens_k).cumsum(0)), dtype=torch.int32, device="cuda")
q = torch.randn(sum(lens_q), 8, 128, device="cuda", dtype=torch.bfloat16)
k = torch.randn(sum(lens_k), 2, 128, device="cuda", dtype=torch.bfloat16)
v = torch.randn(sum(lens_k), 2, 128, device="cuda", dtype=torch.bfloat16)
out, lse = flash_attn_varlen(q, k, v, cq, ck, causal, max_seqlen_q=max(lens_q), return_lse=True, one_launch=True)
loop, lse2 = flash_attn_varlen(q, k, v, cq, ck, causal, return_lse=True, one_launch=False)
torch.cuda.synchronize()
for i in range(len(lens_q)):
    a, b, c, d = int(cq[i]), int(cq[i + 1]), int(ck[i]), int(ck[i + 1])
    ref, ref_lse = flash_attn_reference(q[None, a:b], k[None, c:d], v[None, c:d], causal)
    torch.testing.assert_close(out[a:b].float(), ref[0], atol=2e-2, rtol=2e-2)
    torch.testing.assert_close(lse[:, a:b], ref_lse[0], atol=2e-2, rtol=1e-2)
torch.testing.assert_close(out.float(), loop.float(), atol=2e-2, rtol=2e-2)
torch.testing.assert_close(lse, lse2, atol=2e-2, rtol=1e-2)
# padded KV cache as a packed tensor (what the opt-in one-launch prefill of TP_Attn uses)
B, S, max_len = 3, 130, 512
q2 = torch.randn(B * S, 8, 128, device="cuda", dtype=torch.bfloat16)
k2 = torch.randn(B * max_len, 2, 128, device="cuda", dtype=torch.bfloat16)
v2 = torch.randn(B * max_len, 2, 128, device="cuda", dtype=torch.bfloat16)
ar = torch.arange(B + 1, device="cuda", dtype=torch.int32)
used = torch.tensor([130, 512, 300], device="cuda", dtype=torch.int32)
o2 = flash_attn_varlen(q2, k2, v2, ar * S, ar * max_len, causal, max_seqlen_q=S, one_launch=True, seqused_k=used)
torch.cuda.synchronize()
for b in range(B):
    n = int(used[b])
    ref, _ = flash_attn_reference(q2[None, b * S:(b + 1) * S], k2[None, b * max_len:b * max_len + n], v2[None, b * max_len:b * max_len + n], causal)
    torch.testing.assert_close(o2[b * S:(b + 1) * S].float(), ref[0], atol=2e-2, rtol=2e-2)
print("VARLEN_OK")
"""


@pytest.mark.xfail(strict=False, reason="one-launch varlen instantiation of the flash kernel: compiled, not yet run on hardware")
@pytest.mark.parametrize("causal", [True, False])
def test_flash_varlen_one_launch(causal):
    """cu_seqlens on the device, one launch: against the fp32 reference per sequence and against the per-sequence launches."""
    _isolated(_VARLEN_SNIPPET.format(causal=causal), "VARLEN_OK")


_MEGA_SNIPPET = r"""
import sys, torch
sys.path.insert(0, {root!r})
import triton_dist.utils as U
from triton_dist.mega_kernel import MegaDenseModel
from triton_dist.models import AutoLLM, KV_Cache, ModelConfig
U.initialize_distributed(seed=0)
cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.bfloat16, rank=0, world_size=1)
m = AutoLLM.from_pretrained(cfg)
B = {B}
mk = lambda: KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.bfloat16, 1, "cuda")
kv, kv2 = mk(), mk()
kv.rand_fill_kv_cache(17)
kv2.k_cache.copy_(kv.k_cache); kv2.v_cache.copy_(kv.v_cache); kv2.kv_offset.copy_(kv.kv_offset)
mega = MegaDenseModel(m, B, kv2, attn_splits=2)
for step in range(3):
    ids = torch.randint(0, 1000, (B, 1), device="cuda")
    ref = m.inference(ids, kv.kv_offset.to(torch.int64)[:, None], kv)
    out = mega.mega_forward(ids)
    torch.cuda.synchronize()
    torch.testing.assert_close(out, ref, atol=6e-2, rtol=6e-2)
    kv.inc_offset(1); kv2.inc_offset(1)
print("MEGA_TC_OK")
"""


@pytest.mark.xfail(strict=False, reason="tensor-core LINEAR tasks of the megakernel (mma.sync path for 9..64 tokens): compiled, not yet run on hardware")
@pytest.mark.parametrize("B", [16, 40])
def test_megakernel_tensor_core_linears(B):
    r = subprocess.run([sys.executable, "-c", _MEGA_SNIPPET.format(root=ROOT, B=B)], capture_output=True, text=True, timeout=150, cwd=ROOT)
    assert r.returncode == 0 and "MEGA_TC_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


_MEGA_PAGED_SNIPPET = r"""
import sys, torch
sys.path.insert(0, {root!r})
import triton_dist.utils as U
from triton_dist.mega_kernel import MegaDenseModel
from triton_dist.models import AutoLLM, KV_Cache, ModelConfig, PagedKVCache
U.initialize_distributed(seed=0)
cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.bfloat16, rank=0, world_size=1)
m = AutoLLM.from_pretrained(cfg)
B, ctx_len = 4, 17
kv = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.bfloat16, 1, "cuda")
kv.rand_fill_kv_cache(ctx_len)
paged = PagedKVCache(PAGE_SIZE=8, num_layers=m.num_layers, batch_size=B, max_length=64, num_kv_heads=m.num_key_value_heads,
                     head_dim=m.head_dim, dtype=torch.bfloat16, device="cuda", seed=5)
for li in range(m.num_layers):
    k, v = kv.layer(li)
    paged.append(li, k[:, :ctx_len], v[:, :ctx_len])
paged.inc_offset(ctx_len)
mega = MegaDenseModel(m, B, paged, attn_splits=2)
for step in range(3):
    ids = torch.randint(0, 1000, (B, 1), device="cuda")
    ref = m.inference(ids, kv.kv_offset.to(torch.int64)[:, None], kv)
    out = mega.mega_forward(ids)
    torch.cuda.synchronize()
    torch.testing.assert_close(out, ref, atol=6e-2, rtol=6e-2)
    kv.inc_offset(1); paged.inc_offset(1)
print("MEGA_PAGED_OK")
"""


@pytest.mark.xfail(strict=False, reason="paged-KV task types of the megakernel: exact in the host interpretation, compiled, not yet run on hardware")
def test_megakernel_paged_kv_cache():
    r = subprocess.run([sys.executable, "-c", _MEGA_PAGED_SNIPPET.format(root=ROOT)], capture_output=True, text=True, timeout=150, cwd=ROOT)
    assert r.returncode == 0 and "MEGA_PAGED_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


_PREFILL_SNIPPET = r"""
import sys, torch
sys.path.insert(0, {root!r})
import triton_dist.utils as U
from triton_dist.lk.kernels.flash_mma import run_flash_mma
from triton_dist.mega_kernel import ModelBuilder
U.initialize_distributed(seed=0)
torch.manual_seed(0)
def ref(q, k, v, causal, cap):
    S, G = q.shape[1], q.shape[2] // k.shape[2]
    s = q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 1, 3).repeat_interleave(G, 1).transpose(-1, -2) * 128 ** -0.5
    s = cap * torch.tanh(s / cap) if cap > 0 else s
    if causal:
        s = s.masked_fill(torch.triu(torch.ones(S, S, dtype=torch.bool, device="cuda"), 1), float("-inf"))
    return (torch.softmax(s, -1) @ v.float().permute(0, 2, 1, 3).repeat_interleave(G, 1)).permute(0, 2, 1, 3)
B, S, Hq, Hkv = 2, 333, 8, 2
qkv = torch.randn(B, S, Hq + 2 * Hkv, 128, device="cuda").bfloat16()
q, k, v = qkv[:, :, :Hq], qkv[:, :, Hq:Hq + Hkv], qkv[:, :, Hq + Hkv:]
if {which!r} == "dsl":
    for causal, cap in ((True, 0.0), (False, 4.0)):
        o = run_flash_mma(q, k, v, causal=causal, softcap=cap)
        torch.cuda.synchronize()
        torch.testing.assert_close(o.float(), ref(q, k, v, causal, cap), atol=3e-2, rtol=3e-2)
else:
    mb = ModelBuilder(8)
    out, out2 = torch.zeros(B, S, Hq, 128, device="cuda").bfloat16(), torch.zeros(B, S, Hq, 128, device="cuda").bfloat16()
    d = mb.make_qkv_pack_flash_attn(qkv, out)
    mb.make_flash_attn(q, k, v, out2, is_causal=False, soft_cap=4.0, dep=d)
    mb.compile()
    for _ in range(2):
        mb.run()
    torch.cuda.synchronize()
    torch.testing.assert_close(out.float(), ref(q, k, v, True, 0.0), atol=3e-2, rtol=3e-2)
    torch.testing.assert_close(out2.float(), ref(q, k, v, False, 4.0), atol=3e-2, rtol=3e-2)
print("PREFILL_OK")
"""


@pytest.mark.xfail(strict=False, reason="mma.sync prefill attention (DSL kernel / megakernel FLASH_ATTN task): exact in the CPU interpreter, compiled, not yet run on hardware")
@pytest.mark.parametrize("which", ["dsl", "megakernel"])
def test_prefill_attention_on_mma_sync(which):
    r = subprocess.run([sys.executable, "-c", _PREFILL_SNIPPET.format(root=ROOT, which=which)], capture_output=True, text=True, timeout=200, cwd=ROOT)
    assert r.returncode == 0 and "PREFILL_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


_GDN_SNIPPET = r"""
import torch
from triton_dist.lk.kernels.gdn_chunk import chunk_gated_delta_rule_lk
from triton_dist.ops.gdn import gated_delta_rule_recurrent
T = {T}
torch.manual_seed(T)
B, H, DK, DV = 2, 4, 128, 128
q = (torch.randn(B, T, H, DK, device="cuda") * 0.5).bfloat16()
k = torch.nn.functional.normalize(torch.randn(B, T, H, DK, device="cuda"), dim=-1).bfloat16()
v = (torch.randn(B, T, H, DV, device="cuda") * 0.5).bfloat16()
g, beta = -torch.rand(B, T, H, device="cuda") * 0.3, torch.rand(B, T, H, device="cuda")
s0 = torch.randn(B, H, DK, DV, device="cuda") * 0.1
o, S = chunk_gated_delta_rule_lk(q, k, v, g, beta, initial_state=s0)
torch.cuda.synchronize()
ro, rS = gated_delta_rule_recurrent(q, k, v, g, beta, initial_state=s0)
torch.testing.assert_close(o.float(), ro.float(), atol=3e-2, rtol=3e-2)
torch.testing.assert_close(S, rS, atol=3e-2, rtol=3e-2)
print("GDN_OK")
"""


@pytest.mark.xfail(strict=False, reason="DSL GDN chunk kernels: exact in the CPU interpreter, not yet run on hardware")
@pytest.mark.parametrize("T", [64, 300])
def test_gdn_chunk_dsl_kernels(T):
    _isolated(_GDN_SNIPPET.format(T=T), "GDN_OK")


_PGEMM_SNIPPET = r"""
import torch
from triton_dist.lk.kernels.gemm_sm100 import run_gemm_persistent
torch.manual_seed(0)
for (M, N, K) in ((256, 256, 128), (512, 768, 512), (1000, 392, 320), (4096, 4096, 4096), (8192, 2048, 1024)):
    a = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
    b = (torch.randn(N, K, device="cuda") * 0.5).bfloat16()
    ref = a.float() @ b.float().t()
    c = run_gemm_persistent(a, b)
    torch.cuda.synchronize()
    torch.testing.assert_close(c.float(), ref, atol=0.5, rtol=2e-2)
a = torch.randn(4096, 4096, device="cuda", dtype=torch.bfloat16); b = torch.randn(4096, 4096, device="cuda", dtype=torch.bfloat16)
c = run_gemm_persistent(a, b)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20):
    run_gemm_persistent(a, b, out=c)
e1.record(); torch.cuda.synchronize()
print("lk persistent gemm 4096^3: %.1f us" % (e0.elapsed_time(e1) / 20 * 1e3))
print("PGEMM_OK")
"""


@pytest.mark.xfail(strict=False, reason="persistent rung of the DSL GEMM ladder: compiled and SASS-checked, not yet run on hardware")
def test_lk_gemm_persistent():
    _isolated(_PGEMM_SNIPPET, "PGEMM_OK")


def test_lk_ag_gemm_two_gpus():
    """AllGather + GEMM written in the DSL (comm CTAs + tcgen05 tiles in one kernel); verified across processes in the CPU pipeline
    model, queued for its first hardware run."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["lk_ag_gemm"], nproc=2, timeout=240)


def test_lk_gemm_rs_two_gpus():
    """GEMM + ReduceScatter written in the DSL (tile epilogues reduce into the owner over NVLink, collector CTAs acquire the counter)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["lk_gemm_rs"], nproc=2, timeout=240)


@pytest.mark.xfail(strict=False, reason="megakernel text-generation service: passes on the emulation backend (world 1 / 2), not yet run on hardware")
def test_mega_server_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["mega_server"], nproc=2, timeout=240)


@pytest.mark.xfail(strict=False, reason="OpenSHMEM-style device API from a DSL kernel: passes in the interpreter across processes, compiled, not yet run on hardware")
def test_lk_shmem_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["lk_shmem"], nproc=2, timeout=240)


@pytest.mark.xfail(strict=False, reason="EP dispatch / combine written in the DSL: passes in the interpreter across processes (world 2 / 3), compiled, not yet run on hardware")
def test_lk_ep_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["lk_ep"], nproc=2, timeout=240)


@pytest.mark.xfail(strict=False, reason="megakernel paged-KV tasks with TP-sharded heads: exact on the emulation backend, not yet run on hardware")
def test_mega_paged_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["mega_paged"], nproc=2, timeout=240)


@pytest.mark.xfail(strict=False, reason="Engine.serve(backend='mega'): composition of validated parts, matches the torch backend on the emulation backend, not yet run on hardware")
def test_engine_mega_backend_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist(["engine_mega"], nproc=2, timeout=300)


@pytest.mark.xfail(strict=False, reason="host-level compositions written after the last full hardware session (emulation-tested): variable all-to-all cases, ring copy-engine all-gather producers, packed Ulysses all-to-all")
@pytest.mark.parametrize("case", ["a2a", "allgather_ring", "ulysses_pack", "lk_rs_ring", "lk_ar_tree", "lk_ar_push", "lk_ag_ll", "lk_ar_nvls", "lk_gemm_ar", "allreduce_dsl", "lk_sp_decode", "lk_a2a", "lk_nvls_collectives"])
def test_late_host_level_cases_two_gpus(case):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from _launch import run_dist
    run_dist([case], nproc=2, timeout=150)


@pytest.mark.xfail(strict=False, reason="DSL micro-benchmark suite: kernels verified in the interpreter, first hardware run pending")
def test_lk_microbenchmarks(tmp_path):
    r = subprocess.run([sys.executable, "-m", "triton_dist.lk.bench", "--json", str(tmp_path / "lk_microbench.json")], capture_output=True, text=True,
                       timeout=240, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", "")))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


_DECODE_SNIPPET = r"""
import sys, torch
sys.path.insert(0, {root!r})
from triton_dist.lk.kernels.flash_decode import gqa_decode_lk
from triton_dist.ops.flash_decode import gqa_fwd_batch_decode
torch.manual_seed(0)
B, Hq, Hkv, L = 4, 32, 8, 1024
q = (torch.randn(B, Hq, 128, device="cuda") * 0.5).bfloat16()
k = (torch.randn(B, L, Hkv, 128, device="cuda") * 0.5).bfloat16()
v = (torch.randn(B, L, Hkv, 128, device="cuda") * 0.5).bfloat16()
lens = torch.tensor([1024, 517, 33, 900], device="cuda", dtype=torch.int32)
ref = gqa_fwd_batch_decode(q, k, v, lens)                    # the hardware-validated CUDA kernel
for ns in (1, 8):
    out = gqa_decode_lk(q, k, v, lens, n_splits=ns)
    torch.cuda.synchronize()
    torch.testing.assert_close(out.float(), ref.float(), atol=2e-2, rtol=2e-2)
print("DECODE_OK")
"""


@pytest.mark.xfail(strict=False, reason="DSL decode attention kernels: exact in the interpreter, not yet run on hardware")
def test_lk_decode_attention():
    r = subprocess.run([sys.executable, "-c", _DECODE_SNIPPET.format(root=ROOT)], capture_output=True, text=True, timeout=150, cwd=ROOT)
    assert r.returncode == 0 and "DECODE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]

