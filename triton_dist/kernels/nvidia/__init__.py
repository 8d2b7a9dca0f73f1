"""``triton_dist.kernels.nvidia`` -- the reference's op namespace (kernels/nvidia/__init__.py:25-101), re-exported
from :mod:`triton_dist.ops` where the sm_100a implementations live."""
from ...ops.ag_gemm import (AllGatherGEMMTensorParallelContext, ag_gemm, ag_gemm_mxfp8, create_ag_gemm_context, gemm_non_persistent,  # noqa: F401
                            gemm_persistent)
from ...ops.allgather import (AllGatherMethod, cp_engine_producer_all_gather_inter_node,  # noqa: F401
                              cp_engine_producer_all_gather_intra_node, get_auto_all_gather_method)
from ...ops.comm import (create_fast_allgather_context, fast_allgather, copy_tensor, fill_tensor, reduce_tensor,  # noqa: F401
                         reduce_scatter)
from ...ops.gemm_ar import (create_gemm_ar_context, create_ll_gemm_ar_context, gemm_allreduce_op,  # noqa: F401
                            low_latency_gemm_allreduce_op)
from ...ops.gemm_rs import create_gemm_rs_context, gemm_rs, gemm_rs_mxfp8  # noqa: F401
from ...ops.gemm import gemm as matmul, GemmConfig  # noqa: F401
from ...ops.flash_decode import (gqa_fwd_batch_decode, gqa_fwd_batch_decode_intra_rank,  # noqa: F401
                                 gqa_fwd_batch_decode_persistent)
from ...ops.moe import (ag_group_gemm, create_ag_group_gemm_context, create_moe_ar_context, create_moe_rs_context,  # noqa: F401
                        moe_grouped_gemm, run_moe_reduce_ar, run_moe_reduce_rs)
from ...ops.all_to_all import (all_to_all_post_process, all_to_all_single_2d, all_to_all_vdev_2d, create_all_to_all_context,  # noqa: F401
                               create_all_to_all_single_2d_context, fast_all_to_all)
from ...ops.ep_a2a import combine_kernel_v2, create_ep_ll_a2a_ctx, dispatch_kernel_v2  # noqa: F401
from ...ops.elementwise import swiglu_forward  # noqa: F401
from ...ops.gdn import chunk_gated_delta_rule_fwd  # noqa: F401
from ...parallel.sp import (create_sp_ag_attention_context_intra_node, fused_sp_ag_attn_intra_node)  # noqa: F401
from ...ops.moe import histogram_by_expert as bincount  # noqa: F401
from ...ops.compat import (SpUlysessOAll2AllGemmKernel, SpUlysessQKVGemmAll2AllKernel, UlyssesSpInferPreAttnContext,  # noqa: F401
                           all_to_all_single_gemm, all_to_all_vdev_2d_offset, calc_gather_scatter_index_triton,
                           create_all_to_all_single_gemm_context, create_reduce_scater_2d_ctx,
                           create_ulysses_sp_pre_attn_comm_context, ep_combine_token_inplace, ep_dispatch_token_inplace,
                           fused_sp_ag_attn_inter_node, get_ag_splits_and_recv_offset_for_dispatch, histogram_by_expert_triton,
                           mega_kernel_dispatch_token_moe_grouped_gemm, mega_kernel_moe_grouped_gemm_combine_token,
                           moe_grouped_gemm_2weights, pre_attn_qkv_pack_a2a_op, qkv_bsnd_to_bnsd, reduce_scatter_2d_op,
                           reduce_topk_non_tma, reduce_topk_tma, ring_reduce, swiglu_backward, transposed_moe_grouped_gemm,
                           ulysses_sp_infer_gemm_a2a_op)
from ...ops.perf_model import (estimate_all_gather_time_ms, estimate_gemm_sol_time_ms, estimate_reduce_scatter_time_ms,  # noqa: F401
                               get_dram_gbps, get_nic_gbps_per_gpu, get_tensorcore_tflops)
from ...ops.p2p import p2p_get, p2p_put, p2p_set_signal, p2p_wait_signal  # noqa: F401
from ...ops.gemm_a2a import GemmA2AContext, create_gemm_a2a_context, gemm_all_to_all  # noqa: F401
from ...ops.flash_attn import flash_attn_fwd, flash_attn_varlen  # noqa: F401
from . import allreduce  # noqa: F401
