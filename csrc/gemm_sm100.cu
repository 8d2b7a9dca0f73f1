// Host launcher for the tcgen05 GEMM family (see gemm_sm100.cuh).  C ABI, called from Python via ctypes.
#include "gemm_sm100.cuh"
#include "runtime/driver.h"

using namespace td;
using namespace td::gemm;

// Every field is 8 bytes wide so the ctypes mirror (triton_dist/_C.py: GemmArgs) cannot get padding wrong.
struct TdGemmArgs {
  long long mode;            // 0 plain, 1 AG, 2 RS, 3 AR (rs_* fields: staging / flags / out; rs_rows_per_rank = flag capacity)
  long long is_bf16;         // 1 bf16, 0 fp16, 2 = MXFP8 inputs (e4m3 + UE8M0 scales per 32 K-elements), bf16 output
  long long bn;              // 32 / 64 / 128 / 256
  long long cta_group;       // 1 or 2
  long long group_m;
  long long n_comm_ctas;
  long long use_tma_store;
  long long num_sms;         // CTAs to launch (0 = all SMs)
  long long M, N, K;
  long long m_rot;
  const void* A; long long a_rows; long long lda; long long a_nbuf; long long a_buf_stride_bytes;
  const void* B; long long ldb;
  void* C; long long c_rows; long long ldc; const void* c_phase; long long c_nbuf; long long c_buf_stride_bytes;
  const void* tile_expert; long long num_experts;   // grouped (MoE) mode: B is [num_experts * N, K]
  void* prof_buf; long long prof_cap; long long prof_slots;   // intra-kernel profiler (optional)
  const void* sfa; const void* sfb; long long sfa_chunks; long long sfb_chunks;   // MXFP8: tiled scale factors (512 B chunks)
  // symmetric context
  long long rank, world; unsigned long long symm_base, symm_stride, mc_base;
  void* phase;
  // AG
  long long ag_rows_per_rank, ag_copy_local, ag_skip_wait;   // ag_skip_wait: 1 = GEMM-only twin, 2 = transfer done by the copy engine (1 flag per source), 3 = NVLS multicast push
  const void* ag_a_local; void* ag_ws; long long ag_ws_buf_bytes; void* ag_flags; void* ag_ready;
  // RS
  long long rs_rows_per_rank; void* rs_stage; long long rs_stage_buf_bytes; void* rs_flags; void* rs_out; long long rs_ldo;
  // gather / scatter (MoE grouped GEMM without the gather_rows / scatter_rows passes)
  const void* a_gather; long long a_gather_div; long long a_gather_pad; long long a_src_rows; const void* c_scatter;
  long long expert_stride_rows;   // grouped mode: rows between consecutive experts in B (0 = N); lets a launch use an N-slice of every expert
  // split-K tail (0 / null = off): fp32 scratch + flags (zero-initialised, re-armed by the kernel)
  void* sk_ws; long long sk_ws_bytes; void* sk_flags; long long sk_flag_count; long long sk_max_parts;
  long long rs_skip_wait;         // RS GEMM-only twin
  long long rs_fp32;              // RS ring partial sums in fp32 (staging buffers are [M, N] fp32)
  long long ag_kslices;           // K-sliced AG: K slices (bits 0-7, 0 = default) | comm-CTA groups << 8 | percent of K in the last round << 16
  // mode 4 (MoE reduce-RS / reduce-AR): rs_stage = partial [2][T][N], rs_flags = [2][num_n][W][n_comm], rs_out = output
  const void* row_scale; void* mrs_counter; const void* mrs_total_padded; long long mrs_T, mrs_topk, mrs_allreduce, mrs_chunk_n;
  // mode 5 (Mega-EP dispatch + grouped GEMM): A = ag_ws (symmetric rx [2][rows_cap][K]), flags = ag_flags [2][epr][W][cpd];
  // mode 6 (Mega-EP grouped GEMM + combine): rs_stage = comb [2][pairs][N] symmetric, rs_flags = done [2][W], c_route = return addresses
  const void* epd_send_off; const void* epd_send_ids; const void* epd_dest_off; const void* epd_x;
  long long epd_topk, epd_epr, epd_cpd, epd_rows_cap; void* epd_meta; const void* c_route;
  const void* segk_off; long long segk_n;      // segmented-K batch (mode 0): C is [segk_n][M][N] (c_nbuf / c_buf_stride_bytes)
  const void* scale_a; const void* scale_b;    // fp32 per-row [M] / per-column [N] scales applied in the epilogue (8-bit kinds)
  // AG with 8-bit A: scale_a is then my shard's per-row scale [ag_rows_per_rank]; for MXFP8, sfa / sfa_chunks are the symmetric
  // scale-chunk workspace (both parity halves) and ag_sfa_local my shard's chunks
  void* ag_scale_ws; const void* ag_sfa_local; long long ag_sfa_buf_chunks;
};

static int encode_tmap(CUtensorMap* out, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                       const cuuint32_t* box, int dtype /*0 fp16, 1 bf16, 2 u8, 3 u32 (no swizzle)*/) {
  auto enc = drv::cuTensorMapEncodeTiled_fn();
  if (!enc) { drv::set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return -1; }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUtensorMapDataType dt = dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                 : dtype == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT32;
  CUresult r = enc(out, dt, rank,
                   const_cast<void*>(base), dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   dtype == 3 ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { drv::set_error("cuTensorMapEncodeTiled failed: %s", drv::err_str(r)); return -1; }
  return 0;
}

template <int kMode, int BN, int kCtaGroup, bool kFP8 = false, int kAccStages = 2>
static int launch_cfg(const Params& p, int grid, cudaStream_t stream) {
  // deepest pipeline that fits in 227 KB next to the 32 KB epilogue staging
  constexpr int kStageBytes = SmemLayout<BN, 1, kCtaGroup, 0, kFP8>::kStageBytes;
  constexpr int kMaxStages = (232448 - 1024 - 2 * kCBlockBytes - 384) / kStageBytes;
  constexpr int kStages = kMaxStages > 8 ? 8 : kMaxStages;
  using L = SmemLayout<BN, kStages, kCtaGroup, 0, kFP8>;
  auto kern = gemm_kernel<kMode, BN, kStages, kCtaGroup, kFP8, kAccStages>;
  static bool attr_set = false;
  if (!attr_set) {
    TD_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = L::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = kCtaGroup;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  TD_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p));
  return 0;
}

template <int kMode>
static int dispatch_fp8(const Params& p, int bn, int cg, int grid, cudaStream_t s) {
  if (bn == 128 && cg == 2) return launch_cfg<kMode, 128, 2, true>(p, grid, s);
  if (bn == 128 && cg == 1) return launch_cfg<kMode, 128, 1, true>(p, grid, s);
  // 256-wide tiles halve the L2->SM operand traffic per FLOP (the bf16 kernel is already L2-bound at 64 B/clk/SM);
  // TMEM then holds ONE 256-column accumulator + the scale-factor ring, so the epilogue is not overlapped
  if (bn == 256 && cg == 2) return launch_cfg<kMode, 256, 2, true, 1>(p, grid, s);
  if (bn == 256 && cg == 1) return launch_cfg<kMode, 256, 1, true, 1>(p, grid, s);
  drv::set_error("MXFP8 path supports bn = 128 / 256 (cta_group 1 or 2)");
  return -1;
}

template <int kMode>
static int dispatch(const Params& p, int bn, int cg, int grid, cudaStream_t s) {
#define TD_CASE(BN_, CG_) if (bn == BN_ && cg == CG_) return launch_cfg<kMode, BN_, CG_>(p, grid, s);
  TD_CASE(256, 2) TD_CASE(256, 1) TD_CASE(192, 2) TD_CASE(192, 1) TD_CASE(128, 2) TD_CASE(128, 1)
  TD_CASE(64, 2) TD_CASE(64, 1) TD_CASE(32, 2) TD_CASE(32, 1)
#undef TD_CASE
  drv::set_error("unsupported tile config (bn must be 32/64/128/192/256, cta_group 1/2)");
  return -1;
}

TD_API int td_gemm_launch(const TdGemmArgs* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int cg = static_cast<int>(a->cta_group), bn = static_cast<int>(a->bn);
  const bool fp8 = a->is_bf16 == 2;                            // MXFP8 (block scaled)
  const bool q8 = a->is_bf16 == 3 || a->is_bf16 == 4;          // 3 = int8 x int8 (kind::i8), 4 = e4m3 per-tensor / per-channel scaled
  const int bf16 = (fp8 || q8) ? 2 : (a->is_bf16 != 0 ? 1 : 0);      // tensor-map dtype code of A / B
  const int esz = (fp8 || q8) ? 1 : 2;
  if (a->K % ((fp8 || q8) ? 128 : 8) != 0 || (a->lda * esz) % 16 != 0 || (a->ldb * esz) % 16 != 0) {
    drv::set_error("K must be a multiple of 8 (16-bit) / 128 (MXFP8) and rows 16-byte aligned"); return -1;
  }
  const int bk_elems = (fp8 || q8) ? 128 : BK;
  Params p;
  memset(&p, 0, sizeof(p));
  {  // A: {K, rows, nbuf}
    cuuint64_t dims[3] = {(cuuint64_t)a->K, (cuuint64_t)a->a_rows, (cuuint64_t)(a->a_nbuf > 0 ? a->a_nbuf : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)a->lda * esz, (cuuint64_t)(a->a_nbuf > 1 ? a->a_buf_stride_bytes : a->a_rows * a->lda * esz)};
    cuuint32_t box[3] = {(cuuint32_t)bk_elems, BM, 1};
    if (encode_tmap(&p.tmap_a, a->A, 3, dims, strides, box, bf16)) return -1;
  }
  {  // B: {K, N}
    const long long estride = a->expert_stride_rows > 0 ? a->expert_stride_rows : a->N;
    cuuint64_t dims[2] = {(cuuint64_t)a->K, (cuuint64_t)(a->tile_expert ? (a->num_experts - 1) * estride + a->N : a->N)};
    cuuint64_t strides[1] = {(cuuint64_t)a->ldb * esz};
    cuuint32_t box[2] = {(cuuint32_t)bk_elems, (cuuint32_t)(bn / cg)};
    if (encode_tmap(&p.tmap_b, a->B, 2, dims, strides, box, bf16)) return -1;
  }
  if (a->a_gather) {   // gathered A: {K, source rows}, box {64 elements, 1 row}; one gather4 moves 4 rows x 128 B
    if (cg != 1 || fp8) { drv::set_error("gathered A needs cta_group 1 and 16-bit inputs"); return -1; }
    cuuint64_t dims[2] = {(cuuint64_t)a->K, (cuuint64_t)a->a_src_rows};
    cuuint64_t strides[1] = {(cuuint64_t)a->lda * esz};
    cuuint32_t box[2] = {(cuuint32_t)bk_elems, 1};
    if (encode_tmap(&p.tmap_ag, a->A, 2, dims, strides, box, bf16)) return -1;
    p.a_gather = reinterpret_cast<const int*>(a->a_gather);
    p.a_gather_div = (int)(a->a_gather_div > 0 ? a->a_gather_div : 1); p.a_gather_pad = (int)a->a_gather_pad;
  }
  p.c_scatter = reinterpret_cast<const int*>(a->c_scatter);
  if (!a->a_gather) p.a_gather_pad = (int)a->a_gather_pad;
  p.use_tma_store = (a->use_tma_store && !a->c_scatter && bn >= 64 && a->mode != kRS && a->mode != kAR && a->ldc % 8 == 0) ? 1 : 0;
  if (p.use_tma_store) {  // C: {N, rows, nbuf}
    cuuint64_t dims[3] = {(cuuint64_t)a->N, (cuuint64_t)a->c_rows, (cuuint64_t)(a->c_nbuf > 0 ? a->c_nbuf : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)a->ldc * 2, (cuuint64_t)(a->c_nbuf > 1 ? a->c_buf_stride_bytes : a->c_rows * a->ldc * 2)};
    cuuint32_t box[3] = {kCBlockCols, BM, 1};
    if (encode_tmap(&p.tmap_c, a->C, 3, dims, strides, box, (fp8 || q8) ? 1 : bf16)) return -1;
  }
  p.c_phase = (a->c_nbuf > 1 && !a->segk_off) ? reinterpret_cast<const uint32_t*>(a->c_phase) : nullptr;
  p.c_buf_stride_bytes = a->c_buf_stride_bytes;
  p.tile_expert = reinterpret_cast<const int*>(a->tile_expert);
  p.expert_rows = (int)(a->expert_stride_rows > 0 ? a->expert_stride_rows : a->N);
  p.prof.buf = reinterpret_cast<unsigned long long*>(a->prof_buf); p.prof.cap = (int)a->prof_cap; p.prof.num_slots = (int)a->prof_slots;
  const int TM = BM * cg;
  p.M = (int)a->M; p.N = (int)a->N; p.K = (int)a->K;
  p.num_m = (p.M + TM - 1) / TM;
  p.num_n = (p.N + bn - 1) / bn;
  p.num_k = (p.K + bk_elems - 1) / bk_elems;
  if (fp8) {
    cuuint64_t da[2] = {128, (cuuint64_t)a->sfa_chunks}, db[2] = {128, (cuuint64_t)a->sfb_chunks};
    cuuint64_t st[1] = {512};
    cuuint32_t bx[2] = {128, 1};
    if (encode_tmap(&p.tmap_sfa, a->sfa, 2, da, st, bx, 3)) return -1;
    if (encode_tmap(&p.tmap_sfb, a->sfb, 2, db, st, bx, 3)) return -1;
    if (a->tile_expert) { drv::set_error("MXFP8 grouped GEMM is not wired yet"); return -1; }
  }
  p.group_m = (int)(a->group_m > 0 ? a->group_m : 1);
  if (p.group_m > p.num_m) p.group_m = p.num_m;
  p.m_rot = (int)(((a->m_rot % p.num_m) + p.num_m) % p.num_m);
  p.in_is_bf16 = (a->is_bf16 != 0) ? 1 : 0;      // 16-bit outputs / partial sums are bf16 unless fp16 inputs
  p.in_kind = a->is_bf16 == 3 ? 1 : a->is_bf16 == 4 ? 2 : 0;
  p.bk_elems = bk_elems;
  p.scale_a = reinterpret_cast<const float*>(a->scale_a); p.scale_b = reinterpret_cast<const float*>(a->scale_b);
  if (q8 && (a->mode == kMoeRS || a->mode == kEPD || a->mode == kEPC || a->a_gather)) {
    drv::set_error("8-bit (int8 / e4m3 per-tensor) inputs: plain, ag_gemm, gemm_rs and gemm_ar modes only"); return -1;
  }
  p.ag_esz = esz;
  if (a->mode == kAG && (q8 || fp8) && a->world > 1) {
    if (a->ag_copy_local == 2 || a->ag_skip_wait == 2) {
      drv::set_error("ag_gemm: 8-bit inputs take the in-kernel transports (sm_k / multicast / sm), not copy_engine or all-to-all"); return -1;
    }
    if (a->ag_copy_local != 1 || !a->ag_a_local) { drv::set_error("ag_gemm: 8-bit inputs are pushed from the caller's shard (ag_a_local)"); return -1; }
    if (q8 && a->scale_a && !a->ag_scale_ws) { drv::set_error("ag_gemm: per-row scales of 8-bit A need the scale workspace"); return -1; }
    if (fp8) {
      if (a->ag_rows_per_rank % BM != 0) { drv::set_error("ag_gemm: MXFP8 needs (M / world) %% 128 == 0 (one scale chunk covers 128 rows)"); return -1; }
      if (!a->ag_sfa_local || a->ag_sfa_buf_chunks * 2 != a->sfa_chunks ||
          a->ag_sfa_buf_chunks * BM < (a->ag_ws_buf_bytes / a->K) * (long long)p.num_k) {
        drv::set_error("ag_gemm: MXFP8 needs the scale-chunk workspace [2][max_M / 128][K / 128][512] and the shard's chunks"); return -1;
      }
    }
    p.ag_scale_ws = q8 ? reinterpret_cast<float*>(a->ag_scale_ws) : nullptr;
    p.ag_sf_ws = fp8 ? reinterpret_cast<char*>(const_cast<void*>(a->sfa)) : nullptr;
    p.ag_sf_local = fp8 ? reinterpret_cast<const char*>(a->ag_sfa_local) : nullptr;
    p.ag_sf_buf_chunks = fp8 ? a->ag_sfa_buf_chunks : 0;
  }
  p.n_comm_ctas = (int)a->n_comm_ctas;
  p.C = a->C; p.ldc = a->ldc;
  p.symm.rank = (int)a->rank; p.symm.world = (int)a->world;
  p.symm.base = a->symm_base; p.symm.stride = a->symm_stride; p.symm.mc_base = a->mc_base;
  p.phase = reinterpret_cast<uint32_t*>(a->phase);
  p.ag_rows_per_rank = (int)a->ag_rows_per_rank; p.ag_copy_local = (int)a->ag_copy_local; p.ag_skip_wait = (a->ag_skip_wait == 1) ? 1 : 0;
  p.ag_a_local = a->ag_a_local; p.ag_ws = reinterpret_cast<char*>(a->ag_ws); p.ag_ws_buf_bytes = a->ag_ws_buf_bytes;
  p.ag_flags = reinterpret_cast<uint32_t*>(a->ag_flags); p.ag_ready = reinterpret_cast<uint32_t*>(a->ag_ready);
  p.rs_rows_per_rank = (int)a->rs_rows_per_rank; p.rs_stage = reinterpret_cast<char*>(a->rs_stage);
  p.rs_stage_buf_bytes = a->rs_stage_buf_bytes; p.rs_flags = reinterpret_cast<uint32_t*>(a->rs_flags);
  p.rs_out = a->rs_out; p.rs_ldo = a->rs_ldo;
  p.rs_flag_tiles = (int)a->rs_rows_per_rank;
  if (a->mode == kAR && a->ag_rows_per_rank > 0) {   // scatter flavour borrows the (unused) ag_* fields
    p.a2a_cols_per_rank = (int)a->ag_copy_local; p.a2a_rows_per_src = (int)a->ag_rows_per_rank;
    p.a2a_count = reinterpret_cast<uint32_t*>(a->ag_ready);
  }

  int dev = 0, sms = 0;
  TD_CUDA_CHECK(cudaGetDevice(&dev));
  TD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  int grid = (a->num_sms > 0 && a->num_sms < sms) ? (int)a->num_sms : sms;
  grid -= grid % cg;
  if (p.n_comm_ctas % cg) p.n_comm_ctas += cg - p.n_comm_ctas % cg;
  const int tiles = p.num_m * p.num_n;
  if (a->tile_expert && a->group_m > 1) p.group_m = 1;   // grouped: keep experts' tiles together (n fastest)
  if (a->mode == kAG && a->world > 1 && a->ag_skip_wait == 0) {
    if (p.n_comm_ctas < cg) p.n_comm_ctas = 16;
    if (p.n_comm_ctas > kAGMaxSlices) p.n_comm_ctas = kAGMaxSlices;
  }
  if (a->mode == kAG && a->ag_skip_wait == 2) p.n_comm_ctas = 0;      // copy-engine transport: every SM runs GEMM tiles
  p.ag_nslices = (a->ag_skip_wait == 2) ? 1 : p.n_comm_ctas;
  if (a->mode == kAG && (a->ag_skip_wait == 3 || a->ag_skip_wait == 4)) {
    // K-sliced transports: 3 = NVLS multicast (every rank writes its shard once to the multicast alias), 4 = unicast P2P stores
    // to every peer; both publish one flag per (source, K slice, comm CTA) after ONE release fence per slice
    const bool mcast = a->ag_skip_wait == 3;
    if (mcast && !a->mc_base) { drv::set_error("ag_gemm: multicast transport needs an NVLS multicast mapping"); return -1; }
    if (a->ag_copy_local == 2) { drv::set_error("ag_gemm: the all-to-all flavour cannot use the K-sliced transports"); return -1; }
    if (a->a_gather) { drv::set_error("ag_gemm: the K-sliced transports take dense A"); return -1; }
    if (a->ag_rows_per_rank % BM != 0) { drv::set_error("ag_gemm: K-sliced transports need (M / world) %% 128 == 0"); return -1; }
    if (!mcast && !a->ag_a_local) { drv::set_error("ag_gemm: the P2P K-sliced transport reads the caller's shard (ag_a_local)"); return -1; }
    if (p.n_comm_ctas < cg) p.n_comm_ctas = mcast ? 24 : 32;
    int ks = (int)((a->ag_kslices & 255) > 0 ? (a->ag_kslices & 255) : (mcast ? 8 : 2));
    int groups = (int)((a->ag_kslices >> 8) > 0 ? (a->ag_kslices >> 8) : (mcast ? 3 : 1));
    if (ks > p.num_k) ks = p.num_k;
    if (groups > ks) groups = ks;
    while (groups > 1 && (p.n_comm_ctas % groups != 0 || p.n_comm_ctas / groups < 1)) --groups;
    const int n_c = p.n_comm_ctas / groups;
    while (ks > 1 && n_c * ks > kAGMaxSlices) --ks;
    if (n_c * ks > kAGMaxSlices) { drv::set_error("ag_gemm: too many comm CTAs for the flag array"); return -1; }
    p.ag_multicast = mcast ? 1 : 0;
    p.ag_ctas_per_group = n_c;
    if (ks > 16) ks = 16;
    {  // slice schedule: the comm CTAs work in rounds of `groups` slices that land together; the LAST round carries ~tail_pct
       // of K (what the MMAs still have to do after the last byte), the earlier rounds share the rest evenly
      const int tail_pct = (int)(((a->ag_kslices >> 16) & 255) > 0 ? ((a->ag_kslices >> 16) & 255) : 0);
      const int rounds = (ks + groups - 1) / groups;
      int kb = 0;
      for (int j = 0; j < ks; ++j) {
        p.ag_slice_kb[j] = kb;
        const int round = j / groups, in_round = (round == rounds - 1) ? ks - round * groups : groups;
        double frac;
        if (tail_pct > 0 && rounds > 1) frac = (round == rounds - 1) ? tail_pct / 100.0 / in_round : (1.0 - tail_pct / 100.0) / ((rounds - 1) * groups);
        else frac = 1.0 / ks;
        int n = (int)(frac * p.num_k + 0.5);
        if (n < 1) n = 1;
        const int left = ks - 1 - j;                      // keep at least one k-block for every later slice
        if (kb + n > p.num_k - left) n = p.num_k - left - kb;
        if (j == ks - 1) n = p.num_k - kb;
        kb += n;
      }
      p.ag_slice_kb[ks] = p.num_k;
      p.ag_kslices = ks;
    }
    p.ag_rows_per_cta = (int)((a->ag_rows_per_rank + n_c - 1) / n_c);
    p.ag_nslices = n_c * p.ag_kslices;
  }
  if (a->mode == kAG && a->ag_skip_wait == 0 && p.n_comm_ctas > 0 && a->world <= 4) {
    // few destinations: publish each CTA's share in 4 (TP2) / 2 (TP4) interleaved sub-slices (finer arrival flags)
    int nsub = a->world == 2 ? 4 : 2;
    const size_t shard = (size_t)a->ag_rows_per_rank * a->K * esz;
    while (nsub > 1 && (p.n_comm_ctas * nsub > kAGMaxSlices || shard / (p.n_comm_ctas * nsub) < (64u << 10))) nsub >>= 1;
    p.ag_nslices = p.n_comm_ctas * nsub;
  }
  if (a->mode == kAG && !a->a_gather && a->ag_skip_wait != 2 && a->ag_copy_local != 0 && a->ag_a_local &&
      a->ag_rows_per_rank % BM == 0) {
    // tiles of the local rows are loaded straight from the caller's shard: {K, local rows}, same 64 x 128 box
    const long long lrows = a->ag_copy_local == 2 ? a->ag_rows_per_rank * a->world : a->ag_rows_per_rank;
    cuuint64_t dims[2] = {(cuuint64_t)a->K, (cuuint64_t)lrows};
    cuuint64_t strides[1] = {(cuuint64_t)a->K * esz};
    cuuint32_t box[2] = {(cuuint32_t)bk_elems, BM};
    if (encode_tmap(&p.tmap_al, a->ag_a_local, 2, dims, strides, box, bf16)) return -1;
    if (fp8) {   // and their scale chunks from the caller's tensor: the workspace copy is filled by peers during this launch
      if (!a->ag_sfa_local) { drv::set_error("ag_gemm: MXFP8 needs the shard's scale chunks"); return -1; }
      cuuint64_t ds[2] = {128, (cuuint64_t)(a->ag_rows_per_rank / BM * p.num_k)};
      cuuint64_t st[1] = {512};
      cuuint32_t bx[2] = {128, 1};
      if (encode_tmap(&p.tmap_sfal, a->ag_sfa_local, 2, ds, st, bx, 3)) return -1;
    }
    p.ag_local_direct = 1;
  }
  p.rs_skip_wait = (int)a->rs_skip_wait; p.rs_fp32 = (int)a->rs_fp32;
  p.row_scale = reinterpret_cast<const float*>(a->row_scale);
  if (a->mode == kMoeRS) {
    if (fp8 || !a->c_scatter || !a->tile_expert) { drv::set_error("moe_reduce_rs: needs a 16-bit grouped GEMM with the scatter epilogue"); return -1; }
    if (p.n_comm_ctas < 1 || !a->mrs_counter || !a->mrs_total_padded || !a->rs_stage || !a->rs_flags || !a->rs_out) { drv::set_error("moe_reduce_rs: missing buffers / comm CTAs"); return -1; }
    if (p.N % 8 != 0 || a->rs_ldo % 8 != 0 || a->ldc % 8 != 0) { drv::set_error("moe_reduce_rs: N and row strides must be multiples of 8"); return -1; }
    if (!a->mrs_allreduce && a->mrs_T % a->world != 0) { drv::set_error("moe_reduce_rs: tokens must divide by the world size"); return -1; }
    p.mrs_counter = reinterpret_cast<uint32_t*>(a->mrs_counter); p.mrs_total_padded = reinterpret_cast<const int*>(a->mrs_total_padded);
    p.mrs_T = (int)a->mrs_T; p.mrs_topk = (int)a->mrs_topk; p.mrs_allreduce = (int)a->mrs_allreduce;
    {  // chunk schedule: mrs_chunk_n > 0 = uniform chunks of that many n tiles; 0 = shrinking chunks (~35 % of what is left), so
       // the operand A is re-read only a handful of times while the exposed reduce + pull tail is a single n tile
      int rem = p.num_n, nchunks = 0, start = 0;
      while (rem > 0) {
        int sz = a->mrs_chunk_n > 0 ? (int)a->mrs_chunk_n : (int)(rem * 0.35 + 0.5);
        if (sz < 1) sz = 1;
        if (sz > rem || nchunks == 15) sz = rem;
        p.mrs_chunk_start[nchunks++] = start;
        start += sz; rem -= sz;
      }
      p.mrs_chunk_start[nchunks] = start;
      p.mrs_n_chunks = nchunks;
    }
  }
  if (a->mode == kEPD) {
    if (fp8 || !a->tile_expert || a->a_gather) { drv::set_error("mega_ep dispatch: 16-bit grouped GEMM on the delivered rows"); return -1; }
    if (!a->epd_send_off || !a->epd_send_ids || !a->epd_dest_off || !a->epd_x || !a->epd_meta || !a->ag_ws || !a->ag_flags || a->epd_cpd < 1) {
      drv::set_error("mega_ep dispatch: missing buffers"); return -1;
    }
    p.epd_send_off = (const int*)a->epd_send_off; p.epd_send_ids = (const int*)a->epd_send_ids; p.epd_dest_off = (const int*)a->epd_dest_off;
    p.epd_x = (const char*)a->epd_x; p.epd_topk = (int)a->epd_topk; p.epd_epr = (int)a->epd_epr; p.epd_cpd = (int)a->epd_cpd;
    p.epd_rows_cap = (int)a->epd_rows_cap; p.epd_meta = (uint32_t*)a->epd_meta; p.epd_flags = (uint32_t*)a->ag_flags;
    p.n_comm_ctas = (int)(a->world * a->epd_cpd);
    if (a->K % 8) { drv::set_error("mega_ep dispatch: hidden size must be a multiple of 8"); return -1; }
  }
  if (a->mode == kEPC) {
    if (fp8 || !a->tile_expert || !a->c_route || !a->rs_stage || !a->rs_flags) { drv::set_error("mega_ep combine: missing buffers"); return -1; }
    p.c_route = (const uint32_t*)a->c_route; p.n_comm_ctas = 0; p.use_tma_store = 0;
    if (p.N % 8) { drv::set_error("mega_ep combine: N must be a multiple of 8"); return -1; }
  }
  if (p.n_comm_ctas % cg) p.n_comm_ctas += cg - p.n_comm_ctas % cg;
  if (a->mode == kAR && p.a2a_cols_per_rank > 0) p.n_comm_ctas = 0;     // GEMM + all-to-all: the epilogue scatters, no comm CTAs
  int gemm_ctas = grid - p.n_comm_ctas;      // comm CTAs must be co-resident with the GEMM CTAs: the grid never exceeds the SMs
  if (gemm_ctas < cg) { drv::set_error("no CTAs left for the GEMM (n_comm_ctas too large)"); return -1; }

  // ---- split-K tail: cut the tiles of the last partial wave into K ranges so that idle clusters share them ----
  p.sk_full = tiles; p.sk_rem = 0; p.sk_parts = 1; p.total_units = tiles;
  if (a->sk_ws && a->sk_flags && a->mode != kAR && !a->tile_expert && !a->a_gather && !a->c_scatter) {
    const int workers = gemm_ctas / cg;
    const int full = (tiles / workers) * workers, rem = tiles - full;
    if (rem > 0) {
      int parts = workers / rem;
      if (parts > (int)a->sk_max_parts) parts = (int)a->sk_max_parts;
      while (parts > 1 && p.num_k / parts < 16) --parts;
      const long long need = (long long)rem * (parts - 1) * cg * BM * bn * 4;
      if (parts > 1 && need <= a->sk_ws_bytes && (long long)rem * (parts - 1) * cg <= a->sk_flag_count) {
        p.sk_full = full; p.sk_rem = rem; p.sk_parts = parts; p.total_units = full + rem * parts;
        p.sk_ws = reinterpret_cast<float*>(a->sk_ws); p.sk_flags = reinterpret_cast<uint32_t*>(a->sk_flags);
      }
    }
  }

  if (a->segk_off) {
    if (a->mode != kPlain || a->tile_expert || a->a_gather || fp8 || a->segk_n < 1) { drv::set_error("segmented-K batch: plain 16-bit GEMM only"); return -1; }
    p.segk_off = (const int*)a->segk_off; p.segk_n = (int)a->segk_n; p.segk_tiles = tiles;
    p.sk_full = tiles; p.sk_rem = 0; p.sk_parts = 1; p.sk_ws = nullptr;
    p.total_units = tiles * p.segk_n;
  }
  // never launch more GEMM clusters than work units (idle CTAs would only spin up TMEM)
  if (gemm_ctas / cg > p.total_units) gemm_ctas = p.total_units * cg;
  grid = gemm_ctas + p.n_comm_ctas;

  if (a->mode == kAR) {
    if (fp8) { drv::set_error("gemm_ar: MXFP8 inputs are not wired to the fused all-reduce yet"); return -1; }
    if (p.a2a_cols_per_rank > 0) {
      if (p.a2a_cols_per_rank % bn != 0 || p.a2a_cols_per_rank * p.symm.world != p.N) {
        drv::set_error("gemm_a2a: N must be world * cols_per_rank and cols_per_rank a multiple of the tile width"); return -1;
      }
      if (p.M > p.a2a_rows_per_src) { drv::set_error("gemm_a2a: M exceeds the receive slot"); return -1; }
    } else {
    if (p.n_comm_ctas < cg) { drv::set_error("gemm_ar needs comm CTAs"); return -1; }
    if (p.num_m * cg * p.num_n > p.rs_flag_tiles) { drv::set_error("gemm_ar: flag array too small for this shape"); return -1; }
    }
    if (p.N % 8 != 0 || a->rs_ldo % 8 != 0) { drv::set_error("gemm_ar: N and the output row stride must be multiples of 8"); return -1; }
    if (p.symm.world * cg > 256) { drv::set_error("gemm_ar: world too large"); return -1; }
  }
  if (a->mode == kRS) {
    if (p.rs_rows_per_rank % TM != 0) { drv::set_error("gemm_rs ring path needs (M / world) %% (128 * cta_group) == 0"); return -1; }
    if (p.N % 8 != 0) { drv::set_error("N must be a multiple of 8"); return -1; }
  }
  if (!p.use_tma_store && (a->ldc % 8 != 0 || p.N % 8 != 0)) { drv::set_error("N/ldc must be multiples of 8 elements"); return -1; }
  if (fp8) {
    switch (a->mode) {
      case kPlain: return dispatch_fp8<kPlain>(p, bn, cg, grid, stream);
      case kAG: return dispatch_fp8<kAG>(p, bn, cg, grid, stream);
      case kRS: return dispatch_fp8<kRS>(p, bn, cg, grid, stream);
      default: drv::set_error("bad mode"); return -1;
    }
  }
  switch (a->mode) {
    case kPlain: return dispatch<kPlain>(p, bn, cg, grid, stream);
    case kAG: return dispatch<kAG>(p, bn, cg, grid, stream);
    case kRS: return dispatch<kRS>(p, bn, cg, grid, stream);
    case kAR: return dispatch<kAR>(p, bn, cg, grid, stream);
    case kEPD:
      if (bn == 256 && cg == 2) return launch_cfg<kEPD, 256, 2>(p, grid, stream);
      if (bn == 256 && cg == 1) return launch_cfg<kEPD, 256, 1>(p, grid, stream);
      if (bn == 128 && cg == 2) return launch_cfg<kEPD, 128, 2>(p, grid, stream);
      if (bn == 128 && cg == 1) return launch_cfg<kEPD, 128, 1>(p, grid, stream);
      drv::set_error("mega_ep: bn must be 128 or 256"); return -1;
    case kEPC:
      if (bn == 256 && cg == 2) return launch_cfg<kEPC, 256, 2>(p, grid, stream);
      if (bn == 256 && cg == 1) return launch_cfg<kEPC, 256, 1>(p, grid, stream);
      if (bn == 128 && cg == 2) return launch_cfg<kEPC, 128, 2>(p, grid, stream);
      if (bn == 128 && cg == 1) return launch_cfg<kEPC, 128, 1>(p, grid, stream);
      drv::set_error("mega_ep: bn must be 128 or 256"); return -1;
    case kMoeRS:
      if (bn == 256 && cg == 2) return launch_cfg<kMoeRS, 256, 2>(p, grid, stream);
      if (bn == 256 && cg == 1) return launch_cfg<kMoeRS, 256, 1>(p, grid, stream);
      if (bn == 128 && cg == 2) return launch_cfg<kMoeRS, 128, 2>(p, grid, stream);
      if (bn == 128 && cg == 1) return launch_cfg<kMoeRS, 128, 1>(p, grid, stream);
      drv::set_error("moe_reduce_rs: bn must be 128 or 256"); return -1;
    default: drv::set_error("bad mode"); return -1;
  }
}

// A 2-D tensor map for user (JIT) kernels: row-major [rows, cols] of 1/2/4-byte elements, box {box_inner, box_outer}
TD_API int td_make_tma_2d(void* out_map, const void* base, long long rows, long long cols, long long ld, int elem_bytes, int box_inner,
                          int box_outer, int swizzle) {
  auto enc = drv::cuTensorMapEncodeTiled_fn();
  if (!enc) { drv::set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return -1; }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8;
  const CUtensorMapSwizzle sw = swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(reinterpret_cast<CUtensorMap*>(out_map), dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { drv::set_error("cuTensorMapEncodeTiled failed: %s", drv::err_str(r)); return -1; }
  return 0;
}

TD_API const char* td_last_error() { return td::drv::g_last_error; }
