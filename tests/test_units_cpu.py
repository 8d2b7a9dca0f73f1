"""CPU-only unit tests: build/import, symmetric heap allocator, lazy allocator, autotuner cache, routing sort,
GDN chunked forward, MXFP8 quantisation round trip, single-process model backends, megakernel task graph."""
import math
import os

import pytest
import torch



@pytest.fixture(scope="module")
def dist_env():
    # the emulation backend is forced only for the lifetime of this module's tests: setting it at import time would leak
    # into `pytest -m gpu` runs (pytest imports every test module during collection) and silently put GPU tests on the CPU
    import triton_dist.utils as U
    # GPU tests earlier in the same session may have left the CUDA backend initialised; initialize_distributed would keep it,
    # and the host-protocol tests below (a wait that must time out) would then wait on the device instead
    U.finalize_distributed()
    os.environ.setdefault("MASTER_PORT", "29677")
    os.environ["TD_FORCE_HOST_BACKEND"] = "1"
    U.initialize_distributed(seed=0)
    assert U.current_device().type == "cpu", "dist_env must run on the emulation backend"
    yield U
    U.finalize_distributed()
    os.environ.pop("TD_FORCE_HOST_BACKEND", None)


def test_native_libs_build_and_load():
    from triton_dist import _C
    assert _C.host_lib() is not None
    assert _C.cuda_lib() is not None          # loads without a GPU (driver entry points resolved lazily)
    assert any("libtd_host" in p for p in _C.loaded_libraries())


def test_symmetric_heap_alloc_free(dist_env):
    U = dist_env
    heap = U.get_heap()
    a = U.nvshmem_create_tensor((1000,), torch.float32)
    b = U.nvshmem_create_tensor((3, 5), torch.bfloat16)
    assert heap.contains(a) and heap.contains(b) and a.abs().sum() == 0
    off_a = heap.offset_of(a)
    U.nvshmem_free_tensor_sync(a)
    c = U.nvshmem_create_tensor((10,), torch.int32)
    assert heap.offset_of(c) == off_a                    # first fit reuses the hole
    views = U.nvshmem_create_tensors((4,), torch.int32, U.rank(), 1)
    assert len(views) == 1 and views[0].shape == (4,)
    with pytest.raises(ValueError):
        heap.offset_of(torch.zeros(4))


def test_primitives_host(dist_env):
    from triton_dist import language as dl
    U = dist_env
    sig = U.nvshmem_create_tensor((8,), torch.int32)
    dl.notify(sig[0:1], U.rank(), signal=5, sig_op="set")
    dl.notify(sig[1:2], U.rank(), signal=2, sig_op="add")
    dl.notify(sig[1:2], U.rank(), signal=3, sig_op="add")
    assert sig[0] == 5 and sig[1] == 5
    assert dl.wait(sig[0:2], 2, wait_value=5) == 5
    os.environ["TD_HOST_TIMEOUT_US"] = "20000"
    with pytest.raises(TimeoutError):                    # hang detection instead of spinning forever
        dl.wait(sig[2:3], 1, wait_value=1)
    os.environ.pop("TD_HOST_TIMEOUT_US")
    U.barrier_all_on_stream()


def test_lazy_allocator(dist_env):
    from triton_dist.utils import LazyAllocator
    la = LazyAllocator()
    a = la.declare("a", (100, 7), torch.bfloat16)
    b = la.declare("b", (3,), torch.int64)
    assert la.total_bytes() >= 100 * 7 * 2 + 24 and set(la.breakdown()) == {"a", "b"}
    with pytest.raises(RuntimeError):
        a.get()
    la.materialize()
    assert a.get().shape == (100, 7) and b.get().dtype == torch.int64
    la.free()


def test_autotune_cache(tmp_path, monkeypatch):
    import triton_dist.tune as T
    monkeypatch.setattr(T, "CACHE_DIR", tmp_path)
    calls = []

    @T.autotune([{"k": 1}, {"k": 3}, {"k": 2}], key_fn=lambda x, **kw: str(tuple(x.shape)), warmup=1, rep=2)
    def f(x, config=None):
        calls.append(config["k"])
        import time
        time.sleep(0.002 * config["k"])
        return x * config["k"]

    out = f(torch.ones(4))
    assert out[0] == 1 and f.best_config(torch.ones(4)) == {"k": 1}
    n = len(calls)
    f(torch.ones(4))
    assert len(calls) == n + 1                           # cached: no re-tuning
    assert f(torch.ones(4), autotune=False)[0] == 1


def test_moe_align_sort_and_grouped_gemm_host():
    from triton_dist.ops import moe as M
    torch.manual_seed(0)
    T, topk, E, H, N = 37, 2, 5, 16, 24
    ids = torch.stack([torch.randperm(E)[:topk] for _ in range(T)]).to(torch.int32)
    r = M.moe_align_sort(ids, E, 8)
    flat = r.sorted_ids[r.sorted_ids != r.pad_id]
    assert sorted(flat.tolist()) == list(range(T * topk))
    offs = r.expert_offsets.tolist()
    for e in range(E):
        seg = r.sorted_ids[offs[e]:offs[e + 1]]
        real = seg[seg != r.pad_id]
        assert torch.all(ids.view(-1)[real.long()] == e) and (offs[e + 1] - offs[e]) % 8 == 0
    x = torch.randn(T, H)
    w = torch.randn(E, N, H)
    c = M.moe_forward_local(x, w, ids)
    ref = torch.stack([x[t] @ w[int(ids[t, j])].t() for t in range(T) for j in range(topk)])
    torch.testing.assert_close(c, ref, atol=1e-4, rtol=1e-4)
    wts = torch.rand(T, topk)
    red = M.reduce_topk(c, wts, topk)
    torch.testing.assert_close(red, (ref.view(T, topk, N) * wts[..., None]).sum(1), atol=1e-4, rtol=1e-4)


def test_gdn_chunk_matches_recurrence():
    from triton_dist.ops.gdn import chunk_gated_delta_rule_fwd, gated_delta_rule_recurrent
    torch.manual_seed(0)
    B, T, H, Dk, Dv = 2, 70, 2, 16, 8
    q, k, v = torch.randn(B, T, H, Dk), torch.nn.functional.normalize(torch.randn(B, T, H, Dk), dim=-1), torch.randn(B, T, H, Dv)
    g, beta = -torch.rand(B, T, H) * 0.3, torch.rand(B, T, H)
    o1, s1 = gated_delta_rule_recurrent(q, k, v, g, beta)
    o2, s2 = chunk_gated_delta_rule_fwd(q, k, v, g, beta, chunk_size=16)
    torch.testing.assert_close(o1, o2, atol=1e-4, rtol=1e-4)
    torch.testing.assert_close(s1, s2, atol=1e-4, rtol=1e-4)


def test_mxfp8_roundtrip_and_tiled_scale_layout():
    from triton_dist.ops.fp8 import dequantize_mxfp8, gemm_mxfp8, quantize_mxfp8
    torch.manual_seed(0)
    x = torch.randn(130, 256) * 5
    t = quantize_mxfp8(x)
    assert t.sf.shape == (2, 2, 512)
    d = dequantize_mxfp8(t)
    assert ((d - x).abs() / x.abs().clamp(min=1e-3)).median() < 0.05
    # scale byte of (row 33, k-block 1, chunk 2): chunk (0,1), byte (33 % 32) * 16 + (33 // 32) * 4 + 2
    e = math.ceil(math.log2(x[33, 128 + 64:128 + 96].abs().max().item() / 448.0))
    assert int(t.sf[0, 1, 1 * 16 + 1 * 4 + 2]) == e + 127
    y = gemm_mxfp8(t, quantize_mxfp8(torch.randn(64, 256)))
    assert y.shape == (130, 64)


def test_model_backends_agree_single_process(dist_env):
    from triton_dist.models import Engine, ModelConfig
    for name in ("tiny-dense", "tiny-moe"):
        cfg = ModelConfig(model_name=name, max_length=64, dtype=torch.float32, rank=0, world_size=1)
        eng = Engine(cfg, temperature=0.0)
        ids = torch.randint(0, 1000, (2, 5))
        ref = eng.serve(ids, 4, backend="torch")
        for be in ("triton_dist", "triton_dist_AR"):
            assert torch.equal(eng.serve(ids, 4, backend=be), ref), (name, be)


def test_megakernel_graph_single_process(dist_env):
    from triton_dist.mega_kernel import MegaDenseModel
    from triton_dist.models import AutoLLM, KV_Cache, ModelConfig
    cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.float32, rank=0, world_size=1)
    m = AutoLLM.from_pretrained(cfg)
    B = 2
    kv = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    kv.rand_fill_kv_cache(7)
    kv2 = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    kv2.k_cache.copy_(kv.k_cache); kv2.v_cache.copy_(kv.v_cache); kv2.kv_offset.copy_(kv.kv_offset)
    mega = MegaDenseModel(m, B, kv2, schedule="zig_zag")
    ids = torch.randint(0, 1000, (B, 1))
    ref = m.inference(ids, kv.kv_offset.to(torch.int64)[:, None], kv)
    torch.testing.assert_close(mega.mega_forward(ids), ref, atol=1e-4, rtol=1e-4)
    act = mega.builder.get_sm_activity()
    assert act["tasks"] == sum(v for k, v in act.items() if k not in ("tasks", "counters", "ctas"))


def test_megakernel_batches_above_8_use_tensor_core_tiles(dist_env):
    """Decode batches of 9..64 tokens: the LINEAR tasks get tensor-core tile shapes (8-column groups, a power-of-two number of groups
    per tile, 128 KB fragment staging) and the task list still reproduces the per-op model (host interpretation of the same tasks)."""
    from triton_dist.mega_kernel import T_LINEAR, MegaDenseModel
    from triton_dist.models import AutoLLM, KV_Cache, ModelConfig
    cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.float32, rank=0, world_size=1)
    m = AutoLLM.from_pretrained(cfg)
    B = 24
    kv = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    kv.rand_fill_kv_cache(5)
    kv2 = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    kv2.k_cache.copy_(kv.k_cache); kv2.v_cache.copy_(kv.v_cache); kv2.kv_offset.copy_(kv.kv_offset)
    mega = MegaDenseModel(m, B, kv2)
    lin = [t for t in mega.builder.tasks if t.type == T_LINEAR]
    assert lin and all(t.args[3] % 32 == 0 and t.args[6] % 8 == 0 and t.args[6] <= 128 for t in lin)
    assert mega.builder.max_smem >= 128 * 1024 + 256
    ids = torch.randint(0, 1000, (B, 1))
    ref = m.inference(ids, kv.kv_offset.to(torch.int64)[:, None], kv)
    torch.testing.assert_close(mega.mega_forward(ids), ref, atol=1e-4, rtol=1e-4)
    with pytest.raises(AssertionError):
        MegaDenseModel(m, 65, kv2)


def test_bench_reference_arm_reports_unavailable():
    """No GPU here: the reference arm (the reference's own little_kernel sm_100a GEMM at N=1) must say so and exit 0; it also
    stays `unavailable` for N > 1 (the multi-GPU reference ops need the Triton/NVSHMEM stack that cannot be built offline)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and "unavailable" in d
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "8"], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0 and "unavailable" in json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs writes float32 .npy files holding the same seeded sample of rows on every run; --steps must be >= 1."""
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    t = torch.arange(64 * 3, dtype=torch.bfloat16).reshape(64, 3)
    for d in ("a", "b"):
        bench.dump_outputs(torch, str(tmp_path / d), {"x": (t, 8), "y": (t, 100)}, "_rank1")
    a = np.load(tmp_path / "a" / "x_rank1.npy")
    assert a.dtype == np.float32 and a.shape == (8, 3) and np.array_equal(a, np.load(tmp_path / "b" / "x_rank1.npy"))
    rows = (a[:, 0] / 3).astype(np.int64)
    assert (np.diff(rows) > 0).all() and np.array_equal(a, t.float().numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "y_rank1.npy"), t.float().numpy())
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_flash_attn_reference_paths():
    """CPU path of flash_attn_fwd (the golden the GPU kernel is tested against): causal offsets, per-tile positions, LSE."""
    from triton_dist.ops.flash_attn import flash_attn_fwd, flash_attn_reference, flash_attn_varlen
    torch.manual_seed(0)
    q, k, v = torch.randn(2, 130, 4, 128), torch.randn(2, 300, 2, 128), torch.randn(2, 300, 2, 128)
    o, lse = flash_attn_fwd(q, k, v, causal=True, return_lse=True)
    # brute force for one (batch, head, row): query i sits at position 300 - 130 + i
    b, h, i = 1, 3, 17
    pos = 300 - 130 + i
    s = (q[b, i, h] @ k[b, :pos + 1, h // 2].t()) / math.sqrt(128)
    ref = torch.softmax(s, -1) @ v[b, :pos + 1, h // 2]
    torch.testing.assert_close(o[b, i, h], ref, atol=1e-4, rtol=1e-4)
    torch.testing.assert_close(lse[b, h, i], torch.logsumexp(s, -1), atol=1e-4, rtol=1e-4)
    # explicit tile positions reproduce the default layout
    tp = torch.tensor([[170, 298], [170, 298]], dtype=torch.int32)
    o2 = flash_attn_fwd(q, k, v, causal=True, q_tile_pos=tp)
    torch.testing.assert_close(o2, o)
    # varlen = per-sequence calls
    cu = torch.tensor([0, 50, 130])
    ov = flash_attn_varlen(q[0], k[0, :130], v[0, :130], cu, cu)
    o_first, _ = flash_attn_reference(q[0:1, :50], k[0:1, :50], v[0:1, :50], True)
    torch.testing.assert_close(ov[:50], o_first[0], atol=1e-5, rtol=1e-5)


def test_gdn_recurrent_cpu_fallback():
    from triton_dist.ops.gdn import fused_recurrent_gated_delta_rule, gated_delta_rule_recurrent
    torch.manual_seed(1)
    q, k, v = torch.randn(1, 5, 2, 16), torch.randn(1, 5, 2, 16), torch.randn(1, 5, 2, 8)
    g, beta = -torch.rand(1, 5, 2) * 0.1, torch.rand(1, 5, 2)
    o, s = fused_recurrent_gated_delta_rule(q, k, v, g, beta)
    o2, s2 = gated_delta_rule_recurrent(q, k, v, g, beta)
    torch.testing.assert_close(o, o2); torch.testing.assert_close(s, s2)


def test_megakernel_elementwise_tasks(dist_env):
    """make_silu_mul_up / make_add / make_prefetch of the builder (task graph interpreted by the emulation path)."""
    from triton_dist.mega_kernel import ModelBuilder
    B, inter = 3, 64
    mb = ModelBuilder(B, num_sms=4)
    x = torch.randn(B, 2 * inter)
    act, r, out = torch.zeros(B, inter), torch.randn(B, inter), torch.zeros(B, inter)
    w = torch.randn(256, 64)
    d = mb.make_prefetch(w)
    d = mb.make_silu_mul_up(x, act, dep=d)
    mb.make_add(act, r, out, dep=d)
    mb.compile().run()
    ref = torch.nn.functional.silu(x[:, :inter]) * x[:, inter:]
    torch.testing.assert_close(act, ref)
    torch.testing.assert_close(out, ref + r)


def test_jit_compile_user_kernel():
    """A user kernel written against the device header compiles for sm_100a (no GPU needed) and exports its launcher."""
    from triton_dist.jit import SymmCtx, compile_cuda
    lib = compile_cuda(r"""
        #include "td/primitives.cuh"
        using namespace td;
        __global__ void ring(SymmCtx c, uint32_t* flag, float* data, uint32_t round) {
          const int nxt = (c.rank + 1) % c.world;
          symm_at(c, data, nxt)[threadIdx.x] = c.rank * 100.f + round;
          __syncthreads();
          if (threadIdx.x == 0) notify(c, flag, nxt, round);
          if (threadIdx.x < 32) wait<true, true>(flag, 1, round);
        }
        extern "C" void launch_ring(SymmCtx c, void* flag, void* data, unsigned round, void* stream) {
          ring<<<1, 64, 0, (cudaStream_t)stream>>>(c, (uint32_t*)flag, (float*)data, round);
        }""", name="ring_test")
    assert hasattr(lib, "launch_ring")
    import ctypes
    assert ctypes.sizeof(SymmCtx) == 32


def test_symmetric_heap_fuzz(dist_env):
    """Random allocate / free sequences: live tensors never overlap, stay 256-byte aligned inside the segment, and freeing
    everything returns the heap to one hole (the next big allocation lands at the first offset again)."""
    import random
    U = dist_env
    heap = U.get_heap()
    rng = random.Random(1234)
    probe = U.nvshmem_create_tensor((8,), torch.uint8)
    first = heap.offset_of(probe)
    U.nvshmem_free_tensor_sync(probe)
    live = []
    for step in range(300):
        if live and (rng.random() < 0.45 or len(live) > 40):
            t = live.pop(rng.randrange(len(live)))
            U.nvshmem_free_tensor_sync(t)
        else:
            n = rng.choice([1, 7, 64, 1000, 4096, 100_000])
            t = U.nvshmem_create_tensor((n,), rng.choice([torch.uint8, torch.bfloat16, torch.float32, torch.int64]))
            t.fill_(step % 100)
            live.append(t)
        spans = sorted((heap.offset_of(t), heap.offset_of(t) + t.numel() * t.element_size()) for t in live)
        for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
            assert a1 <= b0, "live symmetric tensors overlap"
        assert all(s[0] % 256 == 0 for s in spans)
    for t in live:
        U.nvshmem_free_tensor_sync(t)
    again = U.nvshmem_create_tensor((1 << 20,), torch.uint8)
    assert heap.offset_of(again) == first
    U.nvshmem_free_tensor_sync(again)


def test_moe_align_sort_properties():
    """Routing invariants for random inputs (emulation path = the specification of the CUDA kernel): every routed pair appears exactly
    once, inside its expert's tile range; unrouted pairs never appear; expert segments are tile aligned."""
    from triton_dist.ops import moe as M
    g = torch.Generator().manual_seed(5)
    for trial in range(20):
        T = int(torch.randint(1, 200, (1,), generator=g))
        E = int(torch.randint(1, 12, (1,), generator=g))
        topk = int(torch.randint(1, min(E, 4) + 1, (1,), generator=g))
        bm = [16, 64, 128][trial % 3]
        ids = torch.stack([torch.randperm(E, generator=g)[:topk] for _ in range(T)]).to(torch.int32)
        ids[torch.rand(T, topk, generator=g) < 0.1] = -1
        r = M.moe_align_sort(ids, E, bm)
        flat = ids.reshape(-1)
        s = r.sorted_ids
        valid = s[s != r.pad_id].long()
        assert sorted(valid.tolist()) == sorted(torch.nonzero(flat >= 0).flatten().tolist())
        assert r.capacity % bm == 0 and all(int(o) % bm == 0 for o in r.expert_offsets)
        for pos in torch.nonzero(s != r.pad_id).flatten().tolist():
            e = int(flat[int(s[pos])])
            assert int(r.expert_offsets[e]) <= pos < int(r.expert_offsets[e + 1])
            assert int(r.tile_expert[pos // bm]) == e


def test_transposed_moe_grouped_gemm_cpu_path():
    """Weight gradient of a grouped GEMM (reference group_gemm.py:988 signature): ragged splits incl. an empty expert, with and
    without the cumulative-offset argument, into a caller-provided buffer."""
    from triton_dist.ops.moe import transposed_moe_grouped_gemm, transpose_gather
    torch.manual_seed(0)
    dy, x = torch.randn(40, 16), torch.randn(40, 24)
    sp = torch.tensor([10, 0, 25, 5])
    ref = torch.stack([dy[0:10].t() @ x[0:10], torch.zeros(16, 24), dy[10:35].t() @ x[10:35], dy[35:40].t() @ x[35:40]])
    torch.testing.assert_close(transposed_moe_grouped_gemm(dy, x, sp), ref)
    buf = torch.full((4, 16, 24), 7.0)
    torch.testing.assert_close(transposed_moe_grouped_gemm(dy, x, sp, torch.cumsum(sp, 0), grad_weight=buf), ref)
    with pytest.raises(TypeError):
        transposed_moe_grouped_gemm(dy, x, sp, bogus_argument=1)
    ids = torch.tensor([3, -1, 0, 39], dtype=torch.int32)
    t = transpose_gather(x, ids, 4)
    assert t.shape == (24, 4) and torch.equal(t[:, 0], x[3]) and torch.all(t[:, 1] == 0) and torch.equal(t[:, 3], x[39])


def test_gemm_scaled_cpu_reference_and_layer_contract():
    """The quantised GEMM's CPU reference path (int8 x per-row / per-channel scales) and the GemmARLayer contract: scales with
    16-bit operands are an error, never silently dropped."""
    from triton_dist.ops.gemm import gemm_scaled
    torch.manual_seed(0)
    a = torch.randint(-127, 128, (6, 32), dtype=torch.int8)
    b = torch.randint(-127, 128, (5, 32), dtype=torch.int8)
    sa, sb = torch.rand(6), torch.rand(5)
    out = gemm_scaled(a, b, sa, sb, out_dtype=torch.float32)
    torch.testing.assert_close(out, (a.float() @ b.float().t()) * sa[:, None] * sb[None, :])
    torch.testing.assert_close(gemm_scaled(a, b, 0.5, None, out_dtype=torch.float32), (a.float() @ b.float().t()) * 0.5)


def test_reference_hint_arguments_are_checked():
    """Reference-only tuning hints are accepted by NAME; anything else raises instead of being swallowed (round-1 `**_unused`)."""
    import triton_dist.utils as U
    U.accept_ref_hints("f", {"BLOCK_M": 128}, ("BLOCK_M", "stages"))
    with pytest.raises(TypeError):
        U.accept_ref_hints("f", {"use_cooperative": True}, ("BLOCK_M",))
    with pytest.raises(NotImplementedError):
        U.accept_ref_hints("f", {"A_scale": torch.ones(1)}, ("A_scale",))


def test_kv_cache_overflow_is_rejected():
    from triton_dist.models import KV_Cache
    kv = KV_Cache(1, 2, 8, 1, 128, torch.float32, 1, "cpu")
    kv.inc_offset(6)
    with pytest.raises(ValueError):
        kv.inc_offset(3)
    kv.clear()
    kv.inc_offset(8)


def test_allreduce_zero_copy_contract():
    """all_reduce may skip its staging copy only for the half the NEXT call reduces (or the stage base under the device-parity
    contract); a stale or offset view of the staging area must raise instead of silently reducing the other half."""
    from triton_dist.ops.comm import AllReduceContext
    ctx = AllReduceContext(1024, 0, 2, 2)
    ctx.stage = torch.zeros(2048, dtype=torch.uint8)
    base = ctx.stage.data_ptr()
    assert ctx.zero_copy_ok(base + 5000, False) is False                 # outside the staging area: ordinary input
    assert ctx.zero_copy_ok(base, True) is True                          # GEMM wrote the device-selected half
    ctx.host_calls = 0                                                   # next call reduces half 1
    assert ctx.zero_copy_ok(base + 1024, False) is True
    with pytest.raises(ValueError):
        ctx.zero_copy_ok(base, False)                                    # stale half
    with pytest.raises(ValueError):
        ctx.zero_copy_ok(base + 1024 + 16, False)                        # offset view
    x = ctx.symm_input(64, torch.float32)
    assert x.data_ptr() == base + 1024


def test_checkpoint_loading_matches_hf_logits(tmp_path):
    """Weight loading (SURVEY 5.4): a HF-format Qwen3 checkpoint written to disk is loaded through ``AutoLLM.from_pretrained``
    (``random_init=False``, local directory: config.json -> ArchConfig, safetensors -> sharded TP weights) and the prefill logits
    match the HF model's own forward."""
    transformers = pytest.importorskip("transformers")
    import triton_dist.utils as U
    from triton_dist.models import AutoLLM, KV_Cache, ModelConfig
    try:
        cfg_hf = transformers.Qwen3Config(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4,
                                          num_key_value_heads=2, head_dim=128, vocab_size=320, max_position_embeddings=128,
                                          tie_word_embeddings=False, rope_theta=1e6)
        torch.manual_seed(0)
        hf = transformers.Qwen3ForCausalLM(cfg_hf).to(torch.float32).eval()
    except Exception as e:      # noqa: BLE001
        pytest.skip(f"transformers cannot build a Qwen3 model here: {e}")
    hf.save_pretrained(str(tmp_path))
    U.initialize_distributed(seed=0)
    mc = ModelConfig(model_name=str(tmp_path), max_length=32, dtype=torch.float32, rank=0, world_size=1, random_init=False)
    m = AutoLLM.from_pretrained(mc)
    assert m.num_layers == 2 and m.head_dim == 128
    ids = torch.randint(0, 320, (2, 7))
    kv = KV_Cache(m.num_layers, 2, 32, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    pos = torch.arange(7)[None, :].expand(2, -1).contiguous()
    logits = m.inference(ids, pos, kv)
    with torch.no_grad():
        ref = hf(ids).logits[:, -1]
    got = logits if logits.dim() == 2 else logits[:, -1]
    torch.testing.assert_close(got.float(), ref.float(), atol=2e-3, rtol=2e-3)


def test_calibrated_perf_models_match_measurements():
    """The round-2 models of the fused kernels (constants from the 8xB200 traces) reproduce the measured times within 15 %."""
    from triton_dist.ops import perf_model as P
    ag = P.estimate_ag_gemm_ms(4096, 512, 4096, 8, "sm_k", 2, 1, 32)
    assert 0.078 < ag < 0.106, ag                  # measured 0.092 ms per call in a back-to-back loop
    rs = P.estimate_gemm_rs_ms(4096, 12288, 6144, 8)
    assert 0.39 < rs < 0.53, rs                    # measured 0.456-0.461 ms
    tr = P.pick_ag_transport(4096, 512, 4096, 8)
    assert tr[0] in ("sm_k", "multicast") and tr[-1] <= ag + 1e-9


def test_gemm_and_collective_models_match_measured_tables():
    """Tile-wave GEMM model vs profiles/README.md section 1 (cta_group 1 sweep) + the round-2 default (cta_group 2), all-reduce fits vs
    section 3, EP dispatch / combine vs section 9: within 15 %; the pickers choose what the measurements chose."""
    import torch
    from triton_dist.ops import perf_model as P
    gemm_us = [((4096, 4096, 4096, 1, 256), 105.5), ((4096, 4096, 4096, 1, 128), 150.0), ((8192, 8192, 8192, 1, 256), 780.0),
               ((8192, 8192, 8192, 1, 128), 1350.0), ((4096, 12288, 6144, 1, 256), 458.0), ((4096, 12288, 6144, 1, 128), 769.0),
               ((8192, 1536, 4096, 1, 256), 87.1), ((8192, 1536, 4096, 1, 128), 138.0), ((4096, 4096, 4096, 2, 256), 88.7),
               ((4096, 12288, 6144, 2, 256), 397.0)]
    for (M, N, K, cg, bn), us in gemm_us:
        est = P.estimate_gemm_ms(M, N, K, cg, bn) * 1e3
        assert 0.85 <= est / us <= 1.15, (M, N, K, cg, bn, est, us)
    assert P.pick_gemm_config(4096, 4096, 4096)[:2] == (2, 256)
    assert P.estimate_gemm_ms(4096, 4096, 4096) >= P.estimate_gemm_sol_time_ms(4096, 4096, 4096) * 0.95      # never (much) below the SOL
    ar_us = [(65536, "OneShot", 34.3), (65536, "TwoShot", 26.8), (65536, "OneShot_Multimem", 22.4), (65536, "TwoShot_Multimem", 23.1),
             (1 << 24, "TwoShot", 103.3), (1 << 24, "OneShot_Multimem", 226.7), (1 << 24, "TwoShot_Multimem", 85.0)]
    for n, m, us in ar_us:
        assert abs(P.estimate_allreduce_us(n, 8, m) - us) / us < 0.05, (n, m)
    assert P.pick_allreduce_method(65536)[0] == "OneShot_Multimem" and P.pick_allreduce_method(1 << 24)[0] == "TwoShot_Multimem"
    assert P.pick_allreduce_method(1 << 24, 8, multimem_ok=False)[0] == "TwoShot"
    assert P.estimate_allreduce_us(1 << 24, 2, "TwoShot") < P.estimate_allreduce_us(1 << 24, 8, "TwoShot")      # less traffic per rank
    assert abs(P.estimate_ep_dispatch_us(128, 7168, 8, 8, 1) - 52.6) / 52.6 < 0.1
    assert abs(P.estimate_ep_dispatch_us(128, 7168, 8, 8, 2) - 71.9) / 71.9 < 0.1
    assert abs(P.estimate_ep_combine_us(128, 7168, 8) - 57.6) / 57.6 < 0.15
    # LL skips the barrier: cheaper for tiny shards, more expensive (2x bytes) for big ones
    assert P.estimate_fast_allgather_us(2048, 8, "push_2d_ll") < P.estimate_fast_allgather_us(2048, 8, "push")
    assert P.estimate_fast_allgather_us(1 << 20, 8, "push_2d_ll") > P.estimate_fast_allgather_us(1 << 20, 8, "push")
    # the reference's signatures (comm_perf_model.py:94-131, gemm_perf_model.py:49-235)
    assert P.estimate_all_gather_time_ms(1 << 30, 8, 8, 770.0, 50.0) == P.estimate_all_gather_time_ms(1 << 30, 8)
    assert P.get_max_tensorcore_tflops(torch.bfloat16, 1965, "NVIDIA B200") == 2250.0
    assert P.get_tensorcore_tflops_by_device_name(torch.float8_e4m3fn, "NVIDIA B200") == 4500.0
    assert P.get_dram_gbps_by_device_name("NVIDIA H800") == 3350.0 and P.get_device_multi_processor_count("B200") == 148
    assert P.get_tflops_approx("B200", 74, 4, torch.bfloat16) == 1125.0


def test_shmem_device_header_compiles_for_sm100a():
    """The NVSHMEM-style device header (csrc/td/shmem.cuh): the self-test kernel of the `shmem` distributed case cross-compiles, and
    the Python mirror's team arithmetic agrees with NVSHMEM's strided-split semantics."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from dist_worker import SHMEM_TEST_SRC
    from triton_dist import jit
    from triton_dist.language.shmem import Team, team_split_strided, team_translate_pe
    lib = jit.compile_cuda(SHMEM_TEST_SRC, name="shmem_selftest")
    assert hasattr(lib, "launch_shmem_selftest")
    world = Team(0, 1, 8)
    even = team_split_strided(world, 0, 2, 4)
    quads = team_split_strided(even, 1, 2, 2)            # members 2 and 6 of the world
    assert even.pes == [0, 2, 4, 6] and quads.pes == [2, 6]
    assert team_translate_pe(quads, 1, world) == 6 and team_translate_pe(world, 6, even) == 3 and team_translate_pe(world, 3, even) == -1
    import pytest
    with pytest.raises(ValueError):
        team_split_strided(world, 4, 2, 3)


def test_flash_attn_varlen_reference_path():
    """Packed variable-length attention (CPU path): per-sequence bottom-right causal masks, LSE in [Hq, Tq] layout."""
    import torch
    from triton_dist.ops.flash_attn import flash_attn_reference, flash_attn_varlen
    torch.manual_seed(0)
    lens_q, lens_k = [5, 130, 0, 64], [9, 130, 4, 200]
    cq = torch.tensor([0] + list(torch.tensor(lens_q).cumsum(0)), dtype=torch.int32)
    ck = torch.tensor([0] + list(torch.tensor(lens_k).cumsum(0)), dtype=torch.int32)
    q, k, v = torch.randn(sum(lens_q), 4, 128), torch.randn(sum(lens_k), 2, 128), torch.randn(sum(lens_k), 2, 128)
    out, lse = flash_attn_varlen(q, k, v, cq, ck, True, return_lse=True)
    assert out.shape == q.shape and lse.shape == (4, sum(lens_q))
    for i in range(len(lens_q)):
        a, b, c, d = int(cq[i]), int(cq[i + 1]), int(ck[i]), int(ck[i + 1])
        if b > a:
            ref, ref_lse = flash_attn_reference(q[None, a:b], k[None, c:d], v[None, c:d], True)
            torch.testing.assert_close(out[a:b], ref[0])
            torch.testing.assert_close(lse[:, a:b], ref_lse[0])
    # a padded KV cache viewed as a packed tensor: slot b holds max_len rows of which seqused_k[b] exist
    B, S, max_len = 3, 5, 20
    q2, k2, v2 = torch.randn(B * S, 4, 128), torch.randn(B * max_len, 2, 128), torch.randn(B * max_len, 2, 128)
    ar, used = torch.arange(B + 1, dtype=torch.int32), torch.tensor([7, 20, 12], dtype=torch.int32)
    o2 = flash_attn_varlen(q2, k2, v2, ar * S, ar * max_len, True, seqused_k=used)
    for b in range(B):
        n = int(used[b])
        ref, _ = flash_attn_reference(q2[None, b * S:(b + 1) * S], k2[None, b * max_len:b * max_len + n], v2[None, b * max_len:b * max_len + n], True)
        torch.testing.assert_close(o2[b * S:(b + 1) * S], ref[0])


def test_paged_kv_cache_feeds_flash_decode():
    """Pages scattered by a random block table: appending through the table and decoding through it equals the dense cache."""
    import math
    import torch
    from triton_dist.models import PagedKVCache
    from triton_dist.ops.flash_decode import _decode_reference, gqa_fwd_batch_decode_partial
    torch.manual_seed(0)
    B, Hq, Hkv, D, L = 3, 4, 2, 128, 2
    cache = PagedKVCache(PAGE_SIZE=4, num_layers=L, batch_size=B, max_length=40, num_kv_heads=Hkv, head_dim=D, dtype=torch.float32, device="cpu")
    dense_k = torch.zeros(L, B, 40, Hkv, D)
    dense_v = torch.zeros(L, B, 40, Hkv, D)
    for S in (7, 1, 1, 5):                                  # a prefill and a few decode steps
        for layer in range(L):
            k_new, v_new = torch.randn(B, S, Hkv, D), torch.randn(B, S, Hkv, D)
            cache.append(layer, k_new, v_new)
            p0 = int(cache.kv_lens[0])
            dense_k[layer, :, p0:p0 + S], dense_v[layer, :, p0:p0 + S] = k_new, v_new
        cache.inc_offset(S)
    assert int(cache.kv_lens[0]) == 14
    q = torch.randn(B, Hq, D)
    for layer in range(L):
        kc, vc, bt, lens = cache.get_layer_kv_cache(layer)
        o, lse = gqa_fwd_batch_decode_partial(q, kc, vc, lens, block_table=bt)
        ro, rl = _decode_reference(q, dense_k[layer], dense_v[layer], lens, 1.0 / math.sqrt(D))
        torch.testing.assert_close(o, ro)
        torch.testing.assert_close(lse, rl)
        gk, gv = cache.gather_dense(layer)
        torch.testing.assert_close(gk[:, :14], dense_k[layer][:, :14])
    import pytest
    with pytest.raises(ValueError):
        cache.inc_offset(100)
    from triton_dist.mega_triton_kernel.models.paged_kv_cache import PagedKVCache as P2          # the reference's module path
    assert P2 is PagedKVCache


def test_engine_profile_option_writes_a_trace(dist_env, tmp_path):
    """Engine.enable_profile (reference: models/engine.py profiler over the first decode steps): a chrome trace per rank."""
    import os
    import torch
    from triton_dist.models import Engine, ModelConfig
    cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.float32, rank=0, world_size=1)
    eng = Engine(cfg, temperature=0.0)
    ids = torch.randint(0, 1000, (2, 5))
    ref = eng.serve(ids, 5, backend="torch", use_cuda_graph=False)
    eng.enable_profile, eng.profile_steps, eng.profile_dir = True, 2, str(tmp_path)
    out = eng.serve(ids, 5, backend="torch", use_cuda_graph=False)
    assert torch.equal(out, ref)                                        # profiling does not change the tokens
    assert os.path.getsize(eng.last_trace) > 1000 and eng.last_trace.endswith("decode_torch_rank0.json")


def test_reference_utils_helpers(dist_env):
    """The generic helpers of the reference's utils.py (platform predicates, CUDA_CHECK, decorators, dtype sizes, lazy tensor specs)."""
    import torch
    import triton_dist.utils as U
    assert U.is_cuda() and not U.is_hip() and not U.is_maca() and U.get_shmem_backend() == "td_symm_heap"
    assert U.is_shmem_initialized() and len(U.get_shmem_hash()) == 16 and U.get_shmem_version()
    U.init_nvshmem_by_torch_process_group(None)
    U.CUDA_CHECK(0); U.CUDA_CHECK((0, "payload"))
    with pytest.raises(RuntimeError):
        U.CUDA_CHECK(700)
    assert U.get_dtype_size(torch.bfloat16) == 2 and U.get_dtype_size(torch.int64) == 8 and U.is_fp8_dtype(torch.float8_e4m3fn)
    assert U.get_device_max_shared_memory_size(0) >= 227 * 1024 and U.support_launch_cooperative_grid()

    @U.requires(lambda: True)
    def ok():
        return 1

    @U.requires(U.is_hip)
    def needs_hip():
        return 2

    assert ok() == 1
    with pytest.raises(AssertionError):
        needs_hip()
    alloc = U.LazyAllocator(symmetric=True)
    lt = alloc.create_tensor((4, 8), torch.float32, name="buf")
    assert isinstance(lt.spec, U.LazyTensorSpec) and lt.spec.nbytes == 128 and U.get_underlying_tensor(lt) is None and not lt.is_materialized
    alloc.materialize()
    assert U.get_underlying_tensor(lt).shape == (4, 8)
    U.nvshmem_free_lazy_tensor(lt)
    assert U.get_underlying_tensor(lt) is None


def test_reference_tooling_names(tmp_path):
    """profiler_utils / tune / autotuner / test.utils helpers a user of the reference expects, with behaviour (not just names)."""
    import json
    import torch
    from triton_dist import autotuner, profiler_utils as PU, tune
    from triton_dist.test.utils import bitwise_equal
    # traces: per-rank processing keeps lanes apart, the parallel dumper writes one valid gzip stream
    tr = {"traceEvents": [{"ph": "X", "pid": 7, "tid": 1, "name": "k", "ts": 0, "dur": 5},
                          {"ph": "M", "pid": 7, "name": "process_name", "args": {"name": "python"}}], "displayTimeUnit": "ms"}
    p1 = PU.process_trace_json(tr, rank=3)
    assert p1["traceEvents"][0]["pid"] == 7 + 3_000_000 and p1["traceEvents"][1]["args"]["name"].startswith("rank 3")
    big = {"traceEvents": [dict(tr["traceEvents"][0], ts=i) for i in range(1234)], "displayTimeUnit": "ms"}
    PU.ParallelJsonDumper(workers=3, chunk_events=100).dump(big, str(tmp_path / "t.json.gz"))
    back = PU.load_json(str(tmp_path / "t.json.gz"))
    assert len(back["traceEvents"]) == 1234 and back["traceEvents"][1233]["ts"] == 1233
    with PU.get_torch_prof_ctx(False) as prof:
        assert prof is None
    with PU.AutoExportProfiler("unit", str(tmp_path), merge=False) as prof:
        torch.ones(8).sum()
    out, ms, peak = PU.benchmark_latency_memory(lambda: torch.ones(16).sum(), 3, 1)
    assert float(out) == 16.0 and ms >= 0 and peak >= 0
    # tune records
    from triton_dist.ops import GemmConfig
    rec = {"cfg": GemmConfig(256, 2, 8, True), "dtype": torch.bfloat16, "t": torch.zeros(2, 3)}
    tune.store_autotune_data(tmp_path / "a" / "rec.json", rec)
    got = tune.load_autotune_data(tmp_path / "a" / "rec.json")
    assert got["cfg"]["bn"] == 256 and got["dtype"] == "torch.bfloat16" and got["t"]["__tensor__"] == [2, 3]
    assert tune.to_hashable({"b": [1, 2], "a": torch.zeros(4)}) == (("a", ("tensor", (4,), "torch.float32")), ("b", (1, 2)))
    assert "bn=256" in tune.pretty_triton_config_repr(GemmConfig(256, 2, 8, True)) and tune.get_hardware_info()["device"]
    assert tune.get_triton_dist_version() and "torch" in tune.get_deps() and set(tune.get_git_info()) == {"commit", "dirty"}
    h = tune.log_to_file(str(tmp_path / "tune.log"))
    tune.log.info("hello")
    h.flush()
    assert "hello" in open(tmp_path / "tune.log").read()
    tune.log.removeHandler(h)
    # contextual autotuner, class form
    calls = []

    def step():
        calls.append(autotuner.override_for("op", "default"))
        return calls[-1]

    t = autotuner.ContextualAutoTuner(step, {"op": ["a", "b"]}, warmup=1, rep=1)
    assert t() in ("a", "b") and t.best["op"] in ("a", "b") and len(t.results) == 2
    x = torch.tensor([0.0, float("nan")])
    assert bitwise_equal(x, x.clone()) and not bitwise_equal(torch.tensor([0.0]), torch.tensor([-0.0]))
    from triton_dist.models.utils import MyLogger
    MyLogger().log("ok", "info")


def test_reference_per_module_names_behave(dist_env):
    """User-facing names of the reference's per-op modules that are thin spellings here: every all-gather method name, the moe_utils
    torch goldens, layer helpers, context-class names."""
    import torch
    from triton_dist.kernels.nvidia import low_latency_allgather as LL
    from triton_dist.kernels.nvidia import moe_utils as MU
    from triton_dist.kernels.nvidia.all_to_all_single_2d import AllToAllSingle2DContext
    from triton_dist.kernels.nvidia.gemm_reduce_scatter import gemm_rs_op  # noqa: F401
    from triton_dist.layers.nvidia.ep_a2a_layer import DispatchCombineContext, EPAllToAllLayoutDesc
    from triton_dist.layers.nvidia.ep_moe import prepare_moe_metadata_using_kernel
    from triton_dist.layers.nvidia.tp_attn import layer_norm
    from triton_dist.layers.nvidia.tp_moe import shard_local
    from triton_dist.ops.all_to_all import AllToAllContext
    assert AllToAllSingle2DContext is AllToAllContext and DispatchCombineContext is EPAllToAllLayoutDesc
    ctx = LL.create_fast_allgather_context(1 << 12)
    x = torch.randn(100)
    for name in ("fast_allgather_pull", "fast_allgather_push_2d", "fast_allgather_push_3d", "fast_allgather_push_2d_ll",
                 "fast_allgather_push_2d_ll_multimem", "fast_allgather_push_numa_2d", "fast_allgather_push_numa_2d_ll"):
        torch.testing.assert_close(getattr(LL, name)(ctx, x).view(-1), x)                 # world 1: the gather is the shard itself
    with pytest.raises(NotImplementedError):
        LL.fast_allgather_push_numa_2d_ll_multinode(ctx, x)
    ctx.finalize()
    ids = torch.tensor([[2, 0], [1, 2], [0, 0]], dtype=torch.int32)
    assert MU.histogram_by_expert_torch(ids, 4).tolist() == [3, 1, 2, 0]
    sc = MU.calc_scatter_index_torch(ids, 4)
    ga = MU.calc_gather_index_torch(ids, 4)
    flat = ids.reshape(-1)
    assert torch.equal(flat[ga.long()], torch.sort(flat, stable=True).values) and torch.equal(ga[sc.reshape(-1).long()], torch.arange(6, dtype=torch.int32))
    h = torch.randn(3, 2, 16)
    w = torch.rand(16) + 0.5
    torch.testing.assert_close(layer_norm(h, w, 1e-6), h * torch.rsqrt(h.pow(2).mean(-1, keepdim=True) + 1e-6) * w, atol=1e-5, rtol=1e-5)
    assert torch.equal(shard_local(torch.arange(12).view(3, 4), 2, 1, 1), torch.tensor([[2, 3], [6, 7], [10, 11]]))
    sorted_ids, tile_expert, offs = prepare_moe_metadata_using_kernel(ids, 4, block_m=4)
    assert offs.numel() == 5 and sorted_ids.numel() % 4 == 0 and tile_expert.numel() == sorted_ids.numel() // 4


def test_megakernel_with_a_paged_kv_cache(dist_env):
    """The megakernel's KV tasks through a block table (T_QKROPE_PAGED / T_ATTN_PAGED): same logits as the dense-cache model, pages
    scattered by a random table, two decode steps (the second reads the token the first one stored through the table)."""
    from triton_dist.mega_kernel import T_ATTN_PAGED, T_QKROPE_PAGED, MegaDenseModel
    from triton_dist.models import AutoLLM, KV_Cache, ModelConfig, PagedKVCache
    cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.float32, rank=0, world_size=1)
    m = AutoLLM.from_pretrained(cfg)
    B, ctx_len = 3, 9
    dense = KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
    dense.rand_fill_kv_cache(ctx_len)
    paged = PagedKVCache(PAGE_SIZE=4, num_layers=m.num_layers, batch_size=B, max_length=64, num_kv_heads=m.num_key_value_heads,
                         head_dim=m.head_dim, dtype=torch.float32, device="cpu", seed=3)
    for li in range(m.num_layers):
        k, v = dense.layer(li)
        paged.append(li, k[:, :ctx_len], v[:, :ctx_len])
    paged.inc_offset(ctx_len)
    mega = MegaDenseModel(m, B, paged, attn_splits=2)
    kinds = {t.type for t in mega.builder.tasks}
    assert T_QKROPE_PAGED in kinds and T_ATTN_PAGED in kinds
    for step in range(2):
        ids = torch.randint(0, 1000, (B, 1))
        ref = m.inference(ids, dense.kv_offset.to(torch.int64)[:, None], dense)
        mega.builder.host_shuffle_seed = step - 1          # latest-ready-first, then a random order: only the scoreboard orders the tasks
        torch.testing.assert_close(mega.mega_forward(ids), ref, atol=1e-4, rtol=1e-4)
        dense.inc_offset(1)
        paged.inc_offset(1)
    gk, _ = paged.gather_dense(0)
    torch.testing.assert_close(gk[:, :ctx_len + 2], dense.layer(0)[0][:, :ctx_len + 2])       # the stored tokens landed in the right pages


def test_megakernel_prefill_tasks(dist_env):
    """Builder ops of the reference's prefill path (make_qkv_pack_qk_norm_rope_split_v -> make_flash_attn, make_qkv_pack_flash_attn) in
    the host interpretation: positions offset by kv_lens, v split out untouched, causal and soft-capped full attention over GQA heads."""
    from triton_dist.mega_kernel import T_FLASH_ATTN, ModelBuilder
    from triton_dist.ops.elementwise import rope_reference
    torch.manual_seed(0)
    B, S, Hq, Hkv = 2, 12, 4, 2
    mb = ModelBuilder(B * S)
    qkv = torch.randn(B, S, Hq + 2 * Hkv, 128).bfloat16()
    kv_lens = torch.tensor([3, 0], dtype=torch.int32)
    qw, kw = torch.rand(128).bfloat16() + 0.5, torch.rand(128).bfloat16() + 0.5
    q_o, k_o, v_o = torch.zeros(B, S, Hq, 128).bfloat16(), torch.zeros(B, S, Hkv, 128).bfloat16(), torch.zeros(B, S, Hkv, 128).bfloat16()
    out, out2 = torch.zeros(B, S, Hq, 128).bfloat16(), torch.zeros(B, S, Hq, 128).bfloat16()
    d = mb.make_qkv_pack_qk_norm_rope_split_v(qkv, kv_lens, qw, kw, q_o, k_o, v_o, 1e-6, 1e6)
    mb.make_flash_attn(q_o, k_o, v_o, out, dep=d)
    mb.make_qkv_pack_flash_attn(qkv, out2, is_causal=False, soft_cap=3.0)
    mb.compile().run()
    assert mb.get_sm_activity()["flash_attn"] == 2 * B * Hq and mb.has_prefill and sum(t.type == T_FLASH_ATTN for t in mb.tasks) == 16

    def ref(q, k, v, causal, cap):
        G = Hq // Hkv
        s = q.float().permute(0, 2, 1, 3) @ k.float().permute(0, 2, 1, 3).repeat_interleave(G, 1).transpose(-1, -2) * 128 ** -0.5
        s = cap * torch.tanh(s / cap) if cap > 0 else s
        if causal:
            s = s.masked_fill(torch.triu(torch.ones(S, S, dtype=torch.bool), 1), float("-inf"))
        return (torch.softmax(s, -1) @ v.float().permute(0, 2, 1, 3).repeat_interleave(G, 1)).permute(0, 2, 1, 3)

    torch.testing.assert_close(out2.float(), ref(qkv[:, :, :Hq], qkv[:, :, Hq:Hq + Hkv], qkv[:, :, Hq + Hkv:], False, 3.0), atol=2e-2, rtol=2e-2)
    torch.testing.assert_close(out.float(), ref(q_o, k_o, v_o, True, 0.0), atol=2e-2, rtol=2e-2)
    assert torch.equal(v_o, qkv[:, :, Hq + Hkv:])
    pos = (kv_lens[:, None] + torch.arange(S)[None]).reshape(-1)
    nrm = lambda z, w: ((z.float() * torch.rsqrt(z.float().pow(2).mean(-1, keepdim=True) + 1e-6)) * w.float()).to(z.dtype)
    torch.testing.assert_close(k_o.view(B * S, Hkv, 128), rope_reference(nrm(qkv[:, :, Hq:Hq + Hkv].reshape(B * S, Hkv, 128), kw), pos, 1e6))


def test_mega_server_single_rank(dist_env):
    """Socket server + client on one rank: JSON-lines protocol, stats, error replies, seeded sampling is reproducible, shutdown."""
    import json
    import threading
    from triton_dist.mega_kernel.server import Client, MegaServer
    srv = MegaServer("tiny-dense", max_length=48, dtype=torch.float32, port=0, max_prompt=16)
    ready = threading.Event()
    th = threading.Thread(target=srv.serve_forever, kwargs=dict(ready=ready), daemon=True)
    th.start()
    assert ready.wait(60)
    try:
        with Client(port=srv.port) as c:
            a = c.request({"prompt_ids": [5, 6, 7], "max_new_tokens": 6, "seed": 11})
            b = c.request({"prompt_ids": [5, 6, 7], "max_new_tokens": 6, "seed": 11})
            assert a["status"] == "success" and a["token_ids"] == b["token_ids"] and a["generated_tokens"] == 6 and a["processing_time"] > 0
            assert c.request({"prompt_ids": list(range(17))})["status"] == "error"           # longer than max_prompt
            assert c.request({"prompt_ids": list(range(1, 17)), "max_new_tokens": 1000})["generated_tokens"] == 48 - 16   # clipped to the cache
            st = c.request({"cmd": "stats"})
            assert st["requests"] == 3 and st["generated_tokens"] == 6 + 6 + 32
            c.f.write(b"not json\n"); c.f.flush()
            assert json.loads(c.f.readline())["status"] == "error"
            assert c.request({"cmd": "shutdown"})["status"] == "success"
    finally:
        th.join(60)
        srv.finalize()
    assert not th.is_alive()


def test_tile_orders_for_arriving_and_leaving_rows():
    """AG + GEMM / GEMM + RS tile orders: permutations; on one node the in-kernel rotations (AG starts at the local shard, RS at rank + 1
    and ends with the own rows); on several nodes the own node first (AG) / last (RS), straddling tiles with the later / earlier node."""
    import numpy as np
    from triton_dist.ops import tile_swizzle as TS
    for (M, W, nn, bm) in ((4096, 8, 1, 128), (4096, 8, 2, 128), (1536, 4, 2, 256), (2048 * 3, 6, 3, 128), (1152, 8, 4, 128)):
        n_tiles = -(-M // bm)
        for r in range(W):
            ag, rs = TS.allgather_gemm_tile_order(M, r, W, nn, bm), TS.gemm_reduce_scatter_tile_order(M, r, W, nn, bm)
            assert sorted(ag.tolist()) == sorted(rs.tolist()) == list(range(n_tiles))
            assert TS.threadblock_swizzle_allgather_gemm_kernel(0, M, r, W, nn, bm) == ag[0]
            assert TS.threadblock_swizzle_gemm_reduce_scatter_kernel(n_tiles - 1, M, r, W, nn, bm) == rs[-1]
            lw, m_rank, m_node = W // nn, M // W, M // nn
            node = r // lw
            # AG: the first tile contains rows of the local shard (or starts right at / after it when the shard is smaller than a tile)
            assert ag[0] * bm < (r + 1) * m_rank and (ag[0] + 1) * bm > r * m_rank or ag[0] * bm >= r * m_rank
            # tiles entirely inside the own node come before any tile entirely inside another node (AG) / after all of them (RS)
            inside = lambda t, n: t * bm >= n * m_node and min(M, (t + 1) * bm) <= (n + 1) * m_node
            own_pos_ag = [i for i, t in enumerate(ag) if inside(t, node)]
            other_pos_ag = [i for i, t in enumerate(ag) if any(inside(t, n) for n in range(nn) if n != node)]
            own_pos_rs = [i for i, t in enumerate(rs) if inside(t, node)]
            other_pos_rs = [i for i, t in enumerate(rs) if any(inside(t, n) for n in range(nn) if n != node)]
            if own_pos_ag and other_pos_ag:
                assert max(own_pos_ag) < min(other_pos_ag) and min(own_pos_rs) > max(other_pos_rs)
            if nn == 1 and m_rank % bm == 0:
                tpr = m_rank // bm
                assert ag.tolist() == [(i + r * tpr) % n_tiles for i in range(n_tiles)]
                assert rs.tolist() == [(i + ((r + 1) % W) * tpr) % n_tiles for i in range(n_tiles)]
    # a tile straddling nodes 0 | 1 (M_node = 576, bm = 128 -> tile 4 holds rows 512..639): AG visits it with the later node, RS with the earlier
    M, W, nn, bm = 1152, 8, 2, 128
    ag0, rs0 = TS.allgather_gemm_tile_order(M, 0, W, nn, bm).tolist(), TS.gemm_reduce_scatter_tile_order(M, 0, W, nn, bm).tolist()
    assert ag0.index(4) >= 4 and set(ag0[:4]) == {0, 1, 2, 3}            # rank 0 (node 0): own-node tiles 0..3 first, the straddler with node 1
    assert rs0.index(4) < 5 and set(rs0[5:]) == {0, 1, 2, 3}              # RS from node 0 visits node 1 first; the straddler goes with it (earlier)
    assert TS.tile_order_table(np.asarray(ag0, dtype=np.int32)).dtype == torch.int32


def test_ep_routing_metadata():
    """get_dispatch_send_reqs / recv_offsets_from_splits against brute force."""
    from triton_dist.ops import ep_metadata as EM
    g = torch.Generator().manual_seed(0)
    W, epr, lw, T, topk = 4, 3, 2, 37, 3
    E = W * epr
    idx = torch.stack([torch.randperm(E, generator=g)[:topk] for _ in range(T)]).to(torch.int32)
    idx[5, 1] = -1                                                                   # a dropped slot
    reqs, counts = EM.get_dispatch_send_reqs(idx, epr, lw, nnodes=W // lw)
    for n in range(W // lw):
        want = [t for t in range(T) if any(0 <= int(e) and int(e) // (epr * lw) == n for e in idx[t])]
        assert reqs[n, :len(want)].tolist() == want and int(counts[n]) == len(want) and (reqs[n, len(want):] == -1).all()
    hist = EM.expert_histogram(idx, E)
    assert int(hist[-1]) == 1 and int(hist.sum()) == T * topk
    full = torch.randint(0, 9, (W, E + 1), generator=g, dtype=torch.int32)
    offs, n_recv, n_in = EM.recv_offsets_from_splits(full, epr)
    for r in range(W):
        run = 0
        for e in range(epr):
            for s in range(W):
                assert int(offs[r, e, s]) == run
                run += int(full[s, r * epr + e])
        assert int(n_recv[r]) == run and int(n_in[r]) == int(full[r, :E].sum())


def test_gemm_config_space_and_matmul_names():
    import importlib
    G = importlib.import_module("triton_dist.ops.gemm")       # ``triton_dist.ops.gemm`` the attribute is the function
    space = G.get_config_space()
    assert len({c.key() for c in space}) == len(space) and {c.bn for c in space} == {32, 64, 128, 192, 256} and {c.cta_group for c in space} == {1, 2}
    assert len(G.get_config_space(persistent=False)) < len(space)
    b = torch.randn(8, 16)
    assert G._as_weight(b).shape == (16, 8) and G._as_weight(b).is_contiguous()
    assert G._as_weight(torch.randn(16, 8).t()).data_ptr() != 0                     # a [K, N] view of an [N, K] weight is used in place
    assert G.matmul_tma_persistent is G.matmul_tma and G.matmul_persistent is G.matmul


def test_host_vector_and_extern_call():
    import ctypes
    from triton_dist import language as dl
    a, b = dl.make_vector([1.0, 2.0, 3.0], torch.float32), dl.zeros_vector(3) + 2.0
    assert ((a + b) * a - 1.0).data.tolist() == [2.0, 7.0, 14.0] and len(a) == 3
    assert a.to(torch.int32).dtype == torch.int32 and a.recast(torch.int32)[0].item() == 0x3F800000
    assert dl.extern_call(ctypes.CDLL(None), "abs", (-5,), restype=ctypes.c_int, argtypes=[ctypes.c_int]) == 5
    from triton_dist.utils import _make_tensor
    t = _make_tensor((4, 4), torch.float32, (0.0, 3.0), device="cpu")
    assert torch.equal(t, torch.full((4, 4), 3.0))


def test_nvml_helpers_degrade_without_a_gpu():
    import importlib
    nv = importlib.import_module("triton_dist.nv_utils")
    raw, eff = nv.calculate_pcie_bandwidth_gbps(5, 16)
    assert raw == 512.0 and abs(eff - 63.0) < 0.1 and nv.calculate_pcie_bandwidth_gbps(2, 8) == (40.0, 4.0)
    assert nv.gpu_uuid_string(bytes(range(16))) == "GPU-00010203-0405-0607-0809-0a0b0c0d0e0f"
    assert nv.get_nvcc().endswith("nvcc") and isinstance(nv.get_physical_device_count(), int)
    assert nv.is_gpu_max_performance_mode(0) in (True, False) and nv.get_pcie_link_max_speed_gbps(0) > 0
    m = nv.get_nvlink_adjacency_matrix()
    assert isinstance(m, list) and nv.has_fullmesh_nvlink_pynvml() in (True, False)
    from triton_dist.utils import _is_cuda_launch_blocking, _torch_has_fp8
    assert _is_cuda_launch_blocking() in (True, False) and _torch_has_fp8()


def test_double_tree_topology_schedulers_and_bookkeeping_helpers():
    from triton_dist.mega_kernel import SchedulingStrategy, enque_tasks, round_robin_scheduler, zig_zag_scheduler
    from triton_dist.ops import comm, perf_model as PM
    from triton_dist.ops.gdn import prepare_chunk_indices, prepare_chunk_offsets, prepare_lens
    from triton_dist.tools.profiler import ProfilerBuffer, decode_tag, parse_to_tracks
    for N in (2, 4, 8, 32):
        trees = [{}, {}]
        for r in range(N):
            t = comm.get_tree_parent_and_children(N, r)
            trees[0][r], trees[1][r] = t[:3], t[3:]
        for T, root in zip(trees, (0, N - 1)):
            seen, stack = set(), [root]
            while stack:
                x = stack.pop()
                assert x not in seen
                seen.add(x)
                for c in T[x][1:]:
                    if c >= 0:
                        assert T[c][0] == x
                        stack.append(c)
            assert seen == set(range(N)) and T[root][0] == -1
        interior = [{r for r in T if T[r][1] >= 0 or T[r][2] >= 0} for T in trees]
        assert not (interior[0] & interior[1])                    # complementary: nobody forwards in both trees
    assert comm.get_max_chunk_nbytes(1 << 20, 8, "oneshot") == 1 << 20
    assert round_robin_scheduler(list(range(7)), 3) == [[0, 3, 6], [1, 4], [2, 5]]
    assert zig_zag_scheduler(list(range(7)), 3) == [[0, 5, 6], [1, 4], [2, 3]]
    assert enque_tasks(list(range(4)), 3, SchedulingStrategy.RUNTIME) == [[0, 1, 2, 3], [], []]
    assert abs(PM.get_tensorcore_tflops_by_calc(torch.bfloat16, clock_rate_mhz=1860.0) - 2255.0) < 5 and "fp8" in PM.get_tensorcore_dtype_support()
    assert PM.get_tensorcore_tflops_by_calc(torch.float8_e4m3fn, clock_rate_mhz=1860.0) == 2 * PM.get_tensorcore_tflops_by_calc(torch.bfloat16, clock_rate_mhz=1860.0)
    assert 60 < PM.get_simd_tflops(torch.float32) < 80
    cu = torch.tensor([0, 5, 5, 70, 134], dtype=torch.int32)
    assert prepare_lens(cu).tolist() == [5, 0, 65, 64]
    assert prepare_chunk_indices(cu, 64).tolist() == [[0, 0], [2, 0], [2, 1], [3, 0]] and prepare_chunk_offsets(cu, 64).tolist() == [0, 1, 1, 3, 4]
    pb = ProfilerBuffer(max_num_profile_slots=16, cap=8, device="cpu")
    ev = lambda tag, start, ns: (tag << 56) | (int(start) << 55) | ns
    pb.buf[9, 0] = 3
    pb.buf[9, 1], pb.buf[9, 2], pb.buf[9, 3] = ev(4, True, 1000), ev(4, False, 3500), ev(5, True, 4000)
    assert decode_tag(ev(4, True, 1000)) == dict(tag=4, start=True, ns=1000)
    tr = parse_to_tracks(pb)
    assert list(tr) == ["cta1.w1"] and tr["cta1.w1"][0]["dur_us"] == 2.5 and tr["cta1.w1"][1]["dur_us"] is None


def test_ag_moe_tile_table_follows_arrival_order():
    """Tiles of the grouped GEMM behind an all-gather: stage ranges match the row order ``moe_align_sort`` produces, execution order is by
    the last shard a tile needs, every tile appears once (uniform, random and many-zero routing)."""
    import numpy as np
    from triton_dist.ops import moe as M
    from triton_dist.ops import tile_swizzle as TS
    g = torch.Generator().manual_seed(0)
    W, E, T, topk, bm = 4, 6, 40, 2, 16
    for kind in ("uniform", "random", "sparse"):
        ids = torch.stack([torch.randperm(E, generator=g)[:topk] for _ in range(W * T)]).to(torch.int32)
        if kind == "uniform":
            ids = (torch.arange(W * T * topk) % E).view(W * T, topk).to(torch.int32)
        if kind == "sparse":
            ids = ids % 2                                                   # most experts receive nothing
        cnt = np.zeros((W, E), dtype=np.int64)
        for s_ in range(W):
            cnt[s_] = np.bincount(ids[s_ * T:(s_ + 1) * T].reshape(-1).numpy(), minlength=E)
        for rank in range(W):
            tab = TS.ag_moe_tile_table(cnt, rank, bm)
            assert TS.check_ag_moe_tile_table(tab, cnt, rank, bm), (kind, rank)
            r = M.moe_align_sort(ids, E, bm, tokens_per_rank=T, rank=rank, world=W)
            for e, t, first, last in tab.tolist():                            # the rows the sort put into that tile come from those stages
                rows = r.sorted_ids[int(r.expert_offsets[e]) + t * bm:int(r.expert_offsets[e]) + (t + 1) * bm]
                rows = rows[rows != r.pad_id]
                stages = ((rows // topk) // T - rank) % W
                assert int(stages.min()) == first and int(stages.max()) == last, (kind, rank, e, t)
    assert not TS.check_swizzled(tab[::-1].copy(), cnt, rank, bm) or len(set(tab[:, 3].tolist())) == 1


def test_megakernel_dependency_graph_under_out_of_order_execution(dist_env):
    """The scoreboard is all the GPU guarantees: the host interpretation can run the tasks in random (or adversarial: latest-ready-first)
    order subject to the counters only.  The dense model's hand-written dependencies and the inferred ones (``auto_deps=True``: storage
    overlap, JOIN tasks for several producers) must give program-order results; a graph with a dependency removed must not."""
    from triton_dist.mega_kernel import T_JOIN, MegaDenseModel, ModelBuilder
    from triton_dist.models import AutoLLM, KV_Cache, ModelConfig
    cfg = ModelConfig(model_name="tiny-dense", max_length=64, dtype=torch.float32, rank=0, world_size=1)
    m = AutoLLM.from_pretrained(cfg)
    for B, fuse, splits in ((2, True, 2), (12, False, 3)):
        mk = lambda: KV_Cache(m.num_layers, B, 64, m.num_key_value_heads, m.head_dim, torch.float32, 1, "cpu")
        kv, kv2 = mk(), mk()
        kv.rand_fill_kv_cache(9)
        kv2.k_cache.copy_(kv.k_cache); kv2.v_cache.copy_(kv.v_cache); kv2.kv_offset.copy_(kv.kv_offset)
        mega = MegaDenseModel(m, B, kv2, fuse_norm=fuse, attn_splits=splits)
        ids = torch.randint(0, 1000, (B, 1))
        ref = m.inference(ids, kv.kv_offset.to(torch.int64)[:, None], kv)
        for seed in (-1, 0, 1, 2):
            mega.builder.host_shuffle_seed = seed
            torch.testing.assert_close(mega.mega_forward(ids), ref, atol=1e-4, rtol=1e-4)
        mega.finalize()

    Bt, H, I = 4, 64, 96
    torch.manual_seed(0)

    def build(auto, break_dep=False):
        mb = ModelBuilder(Bt, num_sms=4, auto_deps=auto)
        x, w1, w2, nw = torch.randn(Bt, H), torch.randn(2 * I, H) * 0.1, torch.randn(H, I) * 0.1, torch.rand(H) + 0.5
        xn, gu, act, y, z = torch.zeros(Bt, H), torch.zeros(Bt, 2 * I), torch.zeros(Bt, I), torch.zeros(Bt, H), torch.zeros(Bt, H)
        if auto:
            mb.make_rms_norm(x, nw, xn, 1e-6)
            mb.make_fc1(xn, w1, gu)
            mb.make_silu_mul_up(gu, act)
            mb.make_fc2(act, w2, y)
            mb.make_add(y, x, z)
            mb.make_add(z, xn, y)                   # reads two producers' outputs and overwrites a buffer another op still reads
        else:
            d = mb.make_rms_norm(x, nw, xn, 1e-6)
            d = mb.make_fc1(xn, w1, gu, d)
            d = mb.make_silu_mul_up(gu, act, dep=d)
            d = mb.make_fc2(act, w2, y, None if break_dep else d)
            d = mb.make_add(y, x, z, dep=d)
            mb.make_add(z, xn, y, dep=d)
        mb.compile()
        xnr = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-6) * nw
        g = xnr @ w1.t()
        return mb, y, (torch.nn.functional.silu(g[:, :I]) * g[:, I:]) @ w2.t() + x + xnr

    for auto in (False, True):
        mb, y, want = build(auto)
        assert (sum(t.type == T_JOIN for t in mb.tasks) > 0) == auto
        for seed in (None, -1, 0, 1, 2, 3):
            mb.host_shuffle_seed = seed
            mb.run()
            torch.testing.assert_close(y, want, atol=1e-4, rtol=1e-4)
    bad, y, want = build(False, break_dep=True)
    bad.host_shuffle_seed = -1
    bad.run()
    assert not torch.allclose(y, want, atol=1e-4)            # the missing edge is visible


def test_tuned_entry_points_expose_their_search_spaces(dist_env):
    from triton_dist.ops import ag_gemm as AG
    from triton_dist.ops import gemm_rs as RS
    space = RS.get_gemm_rs_config_space()
    assert {(c["bn"], c["cta_group"]) for c in space} >= {(256, 2), (128, 1)} and len(AG.ag_gemm_config_space()) == len(AG.AG_GEMM_TUNE_SPACE)
    ctx = RS.create_gemm_rs_context(max_M=256, N=384, rank=0, world_size=1, local_world_size=1, output_dtype=torch.float32)
    A, B = torch.randn(256, 64), torch.randn(384, 64)
    assert RS.gemm_rs_prune_fn(dict(bn=256, cta_group=2), A, B.t(), ctx) and not RS.gemm_rs_prune_fn(dict(bn=192, cta_group=2), A, torch.randn(320, 64).t(), ctx)
    assert not RS.gemm_rs_prune_fn(dict(bn=256, cta_group=2), A[:128], B.t(), ctx) and RS.gemm_rs_prune_fn(dict(bn=256, cta_group=1), A[:128], B.t(), ctx)
    assert "tp1" in RS.gemm_rs_key_fn(A, B.t(), ctx)
    out = RS.gemm_rs_tuned(A, B.t(), ctx, autotune=False)
    torch.testing.assert_close(out, A @ B.t(), atol=1e-4, rtol=1e-4)
    ctx.finalize()


def test_sort_topk_ids_align_block_size_metadata():
    from triton_dist.ops import moe as M
    g = torch.Generator().manual_seed(1)
    W, E, T, topk, bm, rank = 4, 5, 24, 2, 8, 2
    ids = torch.stack([torch.randperm(E, generator=g)[:topk] for _ in range(W * T)]).to(torch.int32)
    sorted_ids, expert_idx, tiled_m, seg0, seg1, ntiles = M.sort_topk_ids_align_block_size(ids, E, rank, W, W, bm)
    assert int(ntiles) == expert_idx.numel() == tiled_m.numel() and torch.all(seg1[:-1] <= seg1[1:]) and len(set(tiled_m.tolist())) == tiled_m.numel()
    for e, tm, s0, s1 in zip(expert_idx.tolist(), tiled_m.tolist(), seg0.tolist(), seg1.tolist()):
        rows = sorted_ids[tm * bm:(tm + 1) * bm]
        rows = rows[rows != ids.numel()]
        assert rows.numel() > 0 and torch.all(ids.view(-1)[rows.long()] == e)                  # the row block belongs to that expert ...
        stages = ((rows // topk) // T - rank) % W
        assert int(stages.min()) == s0 and int(stages.max()) == s1                             # ... and needs exactly those shards
    _, cnt, _ = M.calc_sorted_gather_index(ids, W, E, bm, rank)
    assert cnt.shape == (W, E) and int(cnt.sum()) == ids.numel()


def test_find_topk_picks_a_covering_set_of_configurations(tmp_path):
    """Greedy best-of-k selection over a slowdown matrix: two complementary specialists beat the single best generalist; filters; CLI."""
    import json
    import numpy as np
    from triton_dist.tools.tune import find_topk as F
    # config A wins small shapes, B wins large ones, C is second everywhere (the best SINGLE choice), D is never competitive
    data = {}
    for i, M in enumerate((128, 256, 512, 4096, 8192, 16384)):
        small = M <= 512
        data[str((M, 4096, 4096))] = [dict(cfg=["A"], ms=1.0 if small else 1.6), dict(cfg=["B"], ms=1.7 if small else 1.0),
                                      dict(cfg=["C"], ms=1.08), dict(cfg=["D"], ms=3.0), dict(cfg=["E"], error="launch failed")]
    cfgs, shapes, S = F.slowdown_matrix(data)
    assert cfgs == [("A",), ("B",), ("C",), ("D",)] and S.shape == (4, 6) and np.allclose(S.min(axis=0), 1.0)
    one, stats1 = F.find_best_topk(S, 1)
    two, stats2 = F.find_best_topk(S, 2)
    assert [cfgs[i] for i in one] == [("C",)] and abs(stats1[0] - 1.08) < 1e-9
    assert {cfgs[i] for i in two} == {("A",), ("B",)} and stats2 == (1.0, 1.0, 1.0, 1.0)
    mm, _ = F.find_best_topk(S, 1, objective="minimax")
    assert cfgs[mm[0]] == ("C",)
    _, shapes_small, _ = F.slowdown_matrix(data, [F.IntFilter([1, 512]), F.IntFilter(None), F.IntFilter(4096)])
    assert len(shapes_small) == 3 and F.parse_range("128-1024-128") == (128, 1024, 128) and F.parse_int_range_args(None, "8-64-8").match(64)
    assert not F.IntFilter(7).match(8) and F.IntFilter(7).is_int()
    p = tmp_path / "r.json"
    p.write_text(json.dumps(data))
    assert F.main([str(p), "--topk", "2", "--M-range", "128-512-128"]) == 0

