// tcgen05 / TMEM / TMA persistent GEMM for sm_100a with in-kernel collectives.
//
//   C[M,N] = A[M,K] * B[N,K]^T      (both operands K-major, bf16 or fp16 in, fp32 accumulate in TMEM)
//
// One kernel template covers the family the reference implements as separate Triton kernels plus host
// copy-engine orchestration:
//   kPlain : local GEMM                     (ref: python/triton_dist/kernels/nvidia/gemm.py:396-875,
//                                                 python/little_kernel/benchmark/gemm_sm100/gemm_level9.py)
//   kAG    : AllGather(A) fused with GEMM   (ref: kernels/nvidia/allgather_gemm.py:200-306 + allgather.py:100-124)
//   kRS    : GEMM fused with ReduceScatter  (ref: kernels/nvidia/gemm_reduce_scatter.py:218-332 + reduce_scatter.py)
//   kAR    : GEMM fused with AllReduce      (ref: kernels/nvidia/gemm_allreduce.py:565-604 kernel_fused_gemm_allreduce):
//            the epilogue stores the partial tile into this rank's symmetric staging buffer and raises flag[tile][me]
//            on every rank; comm CTAs of the same grid wait for all W flags of a tile, multimem.ld_reduce it through
//            the NVSwitch (or sum the peers' copies over P2P) and write the reduced tile to the local output
//   kMoeRS : grouped (MoE) GEMM + weighted top-k reduce + ReduceScatter / AllReduce in ONE kernel
//            (ref: kernels/nvidia/moe_reduce_rs.py:168-246 producer with per-chunk flags, :549-619 consumer;
//             moe_reduce_ar.py:563): tiles run n-tile major; the epilogue scales every row by its routing weight and
//            scatters it to (token, k) order; comm CTAs of the same grid wait for "all m tiles of n tile c done", sum the
//            top-k rows of each token into this rank's symmetric partial, flag the peers, and one chunk later every owner
//            pulls the cross-rank sum of ITS rows with multimem.ld_reduce (NVSwitch adds the W partials in fp32)
//   kEPD   : Mega-EP half 1 -- expert-parallel DISPATCH fused with the grouped (gate/up) GEMM (ref: kernels/nvidia/
//            ep_all2all_fused.py:73-835 tile kernels + :839 mega_dispatch_group_gemm): comm CTAs of the same grid store every routed
//            token row straight into its final, expert-sorted and tile-aligned position of the destination rank's A matrix
//            (positions come from the all-gathered per-expert counts, so there is no receive-side index list, sort or copy) and
//            release one flag per (local expert, source, comm CTA); the tcgen05 tiles of an expert start when its flags are up.
//   kEPC   : Mega-EP half 2 -- grouped (down) GEMM fused with the COMBINE transfer (ref :1020 mega_group_gemm_combine): the epilogue
//            stores every output row straight to its (token, k) slot on the rank that owns the token (return address =
//            source << 24 | pair id, delivered by the dispatch); the last CTA release-flags all ranks.
//
// B200-first design (not a translation of the reference):
//   * warp-specialised CTA: warp0 = TMA producer, warp1 = single-thread tcgen05.mma issuer, warp2 = TMEM
//     allocator, warps4-7 = epilogue (tcgen05.ld -> 16-bit -> swizzled smem -> TMA store or coalesced st.global).
//   * optional CTA pairs (cta_group::2, UMMA 256 x BN x 16) with the B tile split across the pair.
//   * double-buffered TMEM accumulators: the epilogue of tile i overlaps the mainloop of tile i+1.
//   * kAG: "comm CTAs" of the same grid PUSH this rank's A shard into every peer's symmetric workspace over
//     NVLink (coalesced 16-byte stores, one byte-slice per comm CTA, nearest consumer first) and publish one
//     release flag per (source, slice) on the destination; the TMA producer warp of a GEMM CTA acquires the
//     flags of the rows it is about to load.  The reference copies with the host copy engine and signals once
//     per source rank (allgather.py:100-124).
//   * kRS: the reduce-scatter is a ring fused into the epilogue: the tile for owner o is computed by rank
//     o-1 first, pushed (coalesced 16-byte stores over NVLink) into rank o-2's staging buffer, which adds
//     its own TMEM accumulator and forwards, ... until rank o adds the last partial and writes the output.
//     No separate reduction pass, no comm SMs; the reference needs scatter + barrier + ring_reduce kernel
//     (reduce_scatter.py:551-707).
//   * all flags carry monotonically increasing phase numbers kept in device memory: no flag reset, no
//     host barrier between calls, and a captured CUDA graph replays correctly.
#pragma once
#include <type_traits>

#include "td/primitives.cuh"
#include "td/profiler.cuh"

namespace td {
namespace gemm {

constexpr int BM = 128;       // rows of C per CTA (UMMA M = 128 * cta_group)
constexpr int BK = 64;        // 64 x 2 B = one 128-byte swizzle row
constexpr int UMMA_K = 16;    // bf16/fp16
constexpr int kThreads = 256;
constexpr int kEpiWarp0 = 4;  // warps 4..7: TMEM lane quadrant == warp_idx % 4
constexpr int kEpiThreads = 128;
constexpr int kCBlockCols = 64;                       // epilogue staging block: 128 rows x 64 cols (16-bit) = 16 KB
constexpr int kCBlockBytes = BM * kCBlockCols * 2;
constexpr int kAGRowsPerChunk = 128;                  // AG arrival-flag granularity (rows of a source shard)
constexpr int kAGMaxSlices = 256;                     // arrival flags per source rank (comm CTAs x sub-slices / K slices)

enum Mode : int { kPlain = 0, kAG = 1, kRS = 2, kAR = 3, kMoeRS = 4, kEPD = 5, kEPC = 6 };

struct Params {
  CUtensorMap tmap_a;   // dims {K, rows_a, nbuf}, box {64, 128, 1}, SWIZZLE_128B
  CUtensorMap tmap_b;   // dims {K, N},            box {64, BN / cta_group}
  CUtensorMap tmap_c;   // dims {N, rows_c, nbuf}, box {64, 128, 1}, SWIZZLE_128B (only if use_tma_store)
  CUtensorMap tmap_sfa; // MXFP8 only: dims {128 (uint32), m_tiles128 * k_blocks}: one 512-byte scale chunk per (128 rows, K=128)
  CUtensorMap tmap_sfb; // MXFP8 only: same for B (n_tiles128 * k_blocks)
  int M, N, K;
  int num_m, num_n, num_k;   // tile counts; num_m is in units of BM * cta_group rows
  int group_m;               // L2 swizzle band height (in m tiles)
  int m_rot;                 // rotate the m-tile order by this many tiles (rank-dependent arrival order)
  int in_is_bf16;            // 1 = bf16, 0 = fp16 (inputs and 16-bit outputs)
  int in_kind;               // 0 = 16-bit inputs (kind::f16); 1 = int8 x int8 -> int32 (kind::i8); 2 = e4m3 x e4m3 -> fp32 (kind::f8f6f4),
                             // both with 128 K-elements per 128-byte smem row and per-row / per-column dequantisation scales
  int bk_elems;              // K elements per smem row (64 for 16-bit, 128 for the 8-bit kinds)
  const float* scale_a;      // optional fp32 [M] per-row scale of C (8-bit kinds: activation scales)
  const float* scale_b;      // optional fp32 [N] per-column scale of C (8-bit kinds: weight scales)
  int use_tma_store;
  int n_comm_ctas;           // CTAs [gridDim.x - n_comm_ctas, gridDim.x) run the collective
  int pad0;
  void* C;                   // output base (row-major)
  long long ldc;             // leading dimension of C in elements
  // optional device-selected output half: C += ((*c_phase + 1) & 1) * c_buf_stride_bytes.  Lets the GEMM write
  // straight into the parity-double-buffered staging of a following collective inside a replayed CUDA graph.
  const uint32_t* c_phase;
  long long c_buf_stride_bytes;
  // optional grouped (MoE) mode: m-tile t multiplies with expert tile_expert[t]'s weight B[e] (rows
  // [e * expert_rows, (e+1) * expert_rows) of the stacked B); tile_expert[t] < 0 marks an unused padded tile.
  // The token rows are pre-sorted by expert and every expert segment is padded to a multiple of the tile height
  // (csrc/moe_kernels.cu: moe_align_sort), so one m-tile never mixes experts.
  const int* tile_expert;
  int expert_rows;
  int pad3;
  // optional intra-kernel profiler (null = off): slot = blockIdx.x * 8 + warp
  ProfBuf prof;
  SymmCtx symm;
  // ---- phase bookkeeping (device resident so a captured graph replays correctly) ----
  // [0] = number of completed calls on this context, [1] = CTA exit counter, [2] = AG local-copy counter
  uint32_t* phase;
  // ---- AG ----
  int ag_rows_per_rank;      // rows of A owned by each rank
  int ag_copy_local;         // 1: comm CTAs copy a_local -> workspace; 0: caller already wrote the workspace; 2: all-to-all (block d of a_local -> rank d)
  int ag_skip_wait;          // GEMM-only twin: never wait (measures exposed communication)
  int ag_multicast;          // 1: comm CTAs write my shard ONCE to the NVLS multicast alias of the workspace (the switch fans it
                             //    out to every rank), K slice by K slice, and publish flag[me][slice * n_comm + cta] on all ranks
  int ag_kslices;            // multicast: number of K slices (every tile starts after 1/ag_kslices of the transfer and follows it)
  int ag_slice_kb[18];       // first k-block (128 bytes of a row) of every K slice (+ end): the last slices are short, so the work left
                             // after the last byte has landed is a few k-blocks
  int ag_rows_per_cta;       // shard rows pushed by one comm CTA
  int ag_ctas_per_group;     // multicast: comm CTAs form n_comm / this groups; group g pushes K slices g, g + G, ... (a release
                             // fence after NVLink stores costs ~7 us of pure latency: G groups keep G slices in flight)
  int ag_local_direct;       // 1: tiles of my own rows read a_local through tmap_al (no local copy, no flag wait)
  CUtensorMap tmap_al;       // {K, rows of a_local}
  int ag_nslices;            // arrival flags per source rank (= comm CTAs, or 1 when the copy engine does the transfer)
  const void* ag_a_local;    // my shard [rows_per_rank, K]
  char* ag_ws;               // my workspace: 2 buffers of [world * rows_per_rank, K] (symmetric)
  long long ag_ws_buf_bytes; // bytes of one buffer
  uint32_t* ag_flags;        // symmetric: [2][world(src)][kAGMaxSlices] = phase of the call that pushed that slice
  uint32_t* ag_ready;        // [world]: ag_ready[s] >= p  <=>  rank s has its phase-p shard in ITS workspace (symmetric)
  int ag_esz;                // bytes per element of A: 2 (16-bit) or 1 (int8 / e4m3 / MXFP8); a gathered row is K * ag_esz bytes
  int pad4;
  // 8-bit payload that travels with the rows (see ag_push_scales).  scale_a is then MY shard's per-row scale [rows_per_rank]
  float* ag_scale_ws;        // int8 / e4m3: symmetric fp32 [2][rows of one workspace half], gathered per-row activation scales
  char* ag_sf_ws;            // MXFP8: symmetric UE8M0 chunks [2][ag_sf_buf_chunks][512]; tmap_sfa spans both halves
  const char* ag_sf_local;   // MXFP8: my shard's chunks [rows_per_rank / 128][num_k][512] (the caller's tensor, also tmap_sfal)
  long long ag_sf_buf_chunks;
  CUtensorMap tmap_sfal;     // MXFP8, own rows read directly (ag_local_direct): {128 (uint32), chunks of my shard}
  // ---- RS (ring) ----
  int rs_rows_per_rank;      // M / world, multiple of BM * cta_group
  int rs_skip_wait;          // GEMM-only twin: never wait for the partial of rank+1 (adds whatever the staging holds)
  int rs_fp32;               // 1: running partial sums travel in fp32 (one rounding at the owner instead of W-1 roundings)
  int pad2;
  char* rs_stage;            // symmetric: 2 buffers of [M, N] 16-bit running partial sums, written by rank+1
  long long rs_stage_buf_bytes;
  uint32_t* rs_flags;        // symmetric: [2][num_m * num_n], written by rank+1 with the phase number
                             // (kAR: [2][rs_flag_tiles][world], flag[tile][r] = phase once rank r staged that 128-row block)
  int rs_flag_tiles;         // kAR: flag capacity per parity, in (128-row block, n tile) units
  int a2a_cols_per_rank;     // kAR scatter flavour (> 0): output columns [d*c, (d+1)*c) go to rank d, rows land at
                             // me * a2a_rows_per_src (GEMM + all-to-all: Ulysses QKV projection); no comm CTAs
  int a2a_rows_per_src;
  // gather / scatter (MoE): A rows of a tile are fetched by TMA tile::gather4 from arbitrary rows of the source matrix
  // (a_gather[row] = id, source row = id / a_gather_div, id == a_gather_pad -> zero row); C rows are written to
  // c_scatter[row] (generic-store epilogue; < 0 or == pad -> skipped)
  const int* a_gather; int a_gather_div; int a_gather_pad;
  const int* c_scatter;
  CUtensorMap tmap_ag;       // {K, rows} with box {64, 1}
  uint32_t* a2a_count;       // local [world] tile counters (last tile for a destination publishes the flag)
  void* rs_out;              // [rows_per_rank, N] final output (local)
  long long rs_ldo;
  // ---- MoE reduce-RS / reduce-AR (kMoeRS) ----
  const float* row_scale;    // optional: the C row scattered to id is multiplied by row_scale[id] (routing weight) in the epilogue
  uint32_t* mrs_counter;     // local [2][chunks + 1]: finished CTA tiles per chunk (+ CTAs done zeroing); this call's parity counts,
                             // the other parity is zeroed for the next call
  const int* mrs_total_padded;   // device: padded row count of the routing (valid m tiles = *p / 128)
  int mrs_T, mrs_topk, mrs_allreduce;
  int mrs_n_chunks;          // column chunks: tiles run chunk-major, then m, then n inside the chunk (A is re-read once per chunk)
  int mrs_chunk_start[17];   // first n tile of every chunk (+ end); chunks shrink towards the end so the exposed tail is one n tile
  // (partial: rs_stage [2][T][N] 16-bit symmetric; flags: rs_flags [2][num_n][W][n_comm]; output: rs_out / rs_ldo)
  // ---- Mega-EP (kEPD / kEPC) ----
  const int* epd_send_off;   // [E + 1]: my (token, k) pairs sorted by GLOBAL expert
  const int* epd_send_ids;   // pair ids (token * topk + k) in that order
  const int* epd_dest_off;   // [E]: first row of MY rows of that expert inside the destination's sorted A
  const char* epd_x;         // my tokens [T, K] 16-bit
  int epd_topk, epd_epr, epd_cpd, epd_rows_cap;   // cpd = comm CTAs per destination rank (n_comm = world * cpd)
  uint32_t* epd_meta;        // symmetric [2][rows_cap]: return address (source << 24 | pair id) of every delivered row
  uint32_t* epd_flags;       // symmetric [2][epr][world][cpd]: phase once that CTA's rows of the expert have landed
  const uint32_t* c_route;   // kEPC epilogue: C row i goes to rank (v >> 24), row (v & 0xffffff) of rs_stage; 0xffffffff = skip
  // ---- segmented-K batch (weight gradients of a grouped GEMM): batch e multiplies the k-blocks [segk_off[e], segk_off[e+1]) of
  // the SAME A / B matrices (reduction dimension = tokens, one segment per expert) into its own output C[e]
  const int* segk_off;       // device int32 [segk_n + 1] in k-blocks; null = off
  int segk_n, segk_tiles;    // batches, tiles per batch (num_m * num_n)
  // ---- split-K tail: the last partial wave of tiles is cut into sk_parts K ranges that run on otherwise idle clusters;
  // parts > 0 park their fp32 accumulator in sk_ws, part 0 adds them in its epilogue (wave quantisation: 768 tiles on
  // 74 CTA pairs = 10.4 waves -> 10.5 instead of 11)
  int sk_full, sk_rem, sk_parts, total_units;
  float* sk_ws;              // [sk_rem][sk_parts - 1][cta_group][BM * BN] fp32
  uint32_t* sk_flags;        // [sk_rem][sk_parts - 1][cta_group], 0 between launches
};

// one schedulable unit of work: a tile and a K range of it
struct Unit { int tile, kb0, kb1, part, slot, batch; };
TD_DEVICE Unit get_unit(const Params& p, int u) {
  Unit x;
  x.batch = 0;
  if (p.segk_off != nullptr) {
    x.batch = u / p.segk_tiles; x.tile = u - x.batch * p.segk_tiles;
    x.kb0 = p.segk_off[x.batch]; x.kb1 = p.segk_off[x.batch + 1]; x.part = 0; x.slot = -1;
    return x;
  }
  if (u < p.sk_full || p.sk_parts <= 1) { x.tile = u; x.kb0 = 0; x.kb1 = p.num_k; x.part = 0; x.slot = -1; return x; }
  const int i = u - p.sk_full;
  x.slot = i % p.sk_rem; x.part = i / p.sk_rem; x.tile = p.sk_full + x.slot;
  x.kb0 = static_cast<int>(static_cast<long long>(x.part) * p.num_k / p.sk_parts);
  x.kb1 = static_cast<int>(static_cast<long long>(x.part + 1) * p.num_k / p.sk_parts);
  return x;
}

// -------------------------------------------------------------------------------------------------
// shared-memory carve-up (GEMM CTAs)
// -------------------------------------------------------------------------------------------------
constexpr int kSFChunk = 512;   // UE8M0 scales of 128 rows x (K = 128): [32 lanes][4 row groups][4 k-blocks of 32]

template <int BN, int kStages, int kCtaGroup, int kExtra = 0, bool kFP8 = false>
struct SmemLayout {
  static constexpr int kABytes = BM * BK * 2;                 // 16 KB (128 rows x 128 B: 64 bf16 or 128 fp8 along K)
  static constexpr int kBBytes = (BN / kCtaGroup) * BK * 2;   // this CTA's share of the B tile
  static constexpr int kSFABytes = kFP8 ? kSFChunk : 0;                           // my 128 rows of A
  static constexpr int kSFBBytes = kFP8 ? ((BN + 127) / 128) * kSFChunk : 0;      // ALL BN columns (needed by both CTAs)
  static constexpr int kSFPad = kFP8 ? (1024 - (kSFABytes + kSFBBytes) % 1024) % 1024 : 0;
  static constexpr int kStageBytes = kABytes + kBBytes + kSFABytes + kSFBBytes + kSFPad;
  static constexpr int kTxBytes = kABytes + kBBytes + kSFABytes + kSFBBytes;      // bytes one CTA lands per stage
  static constexpr int kCOff = kStages * kStageBytes;
  static constexpr int kBarOff = kCOff + 2 * kCBlockBytes;
  // barriers: full[kStages], empty[kStages], tmem_full[2], tmem_empty[2]; then the TMEM base pointer
  static constexpr int kNumBars = 2 * kStages + 4;
  static constexpr int kExtraOff = ((kBarOff + kNumBars * 8 + 16 + 127) / 128) * 128;   // optional comm ring (AG mode)
  static constexpr int kGemmBytes = kExtraOff + kExtra;
  static constexpr int kTotal = kGemmBytes + 1024;  // + alignment slack (comm CTAs use no shared memory)
  static_assert(kStageBytes % 1024 == 0, "stage must keep 1024 B alignment for SWIZZLE_128B");
  static_assert(kTotal <= 232448, "exceeds 227 KB of shared memory");
};

__host__ __device__ constexpr int tmem_cols_for(int bn) {
  return 2 * bn <= 32 ? 32 : 2 * bn <= 64 ? 64 : 2 * bn <= 128 ? 128 : 2 * bn <= 256 ? 256 : 512;
}

// bytes of my shard pushed by one comm CTA (128-byte aligned slices)
__host__ __device__ inline size_t ag_slice_bytes(size_t shard_bytes, int n_comm) {
  const size_t n = n_comm > 0 ? n_comm : 1;
  return ((shard_bytes + n - 1) / n + 127) & ~static_cast<size_t>(127);
}

// tile index -> (m tile, n tile); band-swizzled (m fastest inside a band of group_m tiles), then rotated
TD_DEVICE void tile_coords(const Params& p, int t, int& m_tile, int& n_tile) {
  if (p.mrs_n_chunks > 0) {     // MoE reduce-RS: chunk of n tiles (outer), m tile, n tile inside the chunk (inner)
    int c = 0, r = t;
    while (c + 1 < p.mrs_n_chunks && r >= p.num_m * (p.mrs_chunk_start[c + 1] - p.mrs_chunk_start[c])) {
      r -= p.num_m * (p.mrs_chunk_start[c + 1] - p.mrs_chunk_start[c]);
      ++c;
    }
    const int cn = p.mrs_chunk_start[c + 1] - p.mrs_chunk_start[c];
    m_tile = r / cn;
    n_tile = p.mrs_chunk_start[c] + r % cn;
    return;
  }
  const int per_band = p.group_m * p.num_n;
  const int band = t / per_band;
  const int first_m = band * p.group_m;
  const int band_m = min(p.num_m - first_m, p.group_m);
  const int r = t - band * per_band;
  n_tile = r / band_m;
  m_tile = first_m + r % band_m + p.m_rot;
  if (m_tile >= p.num_m) m_tile -= p.num_m;
}

// -------------------------------------------------------------------------------------------------
// AG consumer side: wait until rows [row0, row1) of the gathered A are resident in my workspace
// -------------------------------------------------------------------------------------------------
TD_DEVICE void ag_wait_rows(const Params& p, uint32_t ph, int row0, int row1) {
  // The source rank's comm CTA c pushes byte slice c of its shard and then publishes flag[src][c] = phase on the
  // destination.  A flag holds the phase number of the call that last filled it, so stale values from earlier
  // calls (or other shapes) are simply "< ph" and nothing is ever reset.
  const int Ms = p.ag_rows_per_rank;
  const size_t row_bytes = static_cast<size_t>(p.K) * p.ag_esz;
  const size_t shard_bytes = static_cast<size_t>(Ms) * row_bytes;
  const size_t slice = ag_slice_bytes(shard_bytes, p.ag_nslices);
  const uint32_t* flags = p.ag_flags + (ph & 1u) * p.symm.world * kAGMaxSlices;
  int r = row0;
  while (r < row1) {
    const int s = r / Ms;
    const int r_end = min(row1, (s + 1) * Ms);
    if (s != p.symm.rank || (p.ag_copy_local && !p.ag_local_direct)) {
      const size_t b0 = static_cast<size_t>(r - s * Ms) * row_bytes, b1 = static_cast<size_t>(r_end - s * Ms) * row_bytes;
      for (int c = static_cast<int>(b0 / slice); c <= static_cast<int>((b1 - 1) / slice); ++c)
        wait_ge<true>(flags + s * kAGMaxSlices + c, ph);
    }
    r = r_end;
  }
  // rows were written by (remote) generic-proxy stores and are about to be read by TMA (async proxy)
  ptx::fence_proxy_async();
}

// K-sliced (multicast) transport: rows [r_local, r_local + BM) of source s, K slice j.  Comm CTA c of the source pushes rows
// [c * rows_per_cta, (c + 1) * rows_per_cta) of every slice and publishes flag[s][j * n_comm + c].
TD_DEVICE void ag_wait_kslice(const Params& p, uint32_t ph, int s, int r_local, int j) {
  const uint32_t* flags = p.ag_flags + (ph & 1u) * p.symm.world * kAGMaxSlices + s * kAGMaxSlices + j * p.ag_ctas_per_group;
  const int c0 = r_local / p.ag_rows_per_cta;
  const int c1 = (min(r_local + BM, p.ag_rows_per_rank) - 1) / p.ag_rows_per_cta;
  for (int c = c0; c <= c1; ++c) wait_ge<true>(flags + c, ph);
  ptx::fence_proxy_async();
}

// -------------------------------------------------------------------------------------------------
// AG producer side (comm CTA c): PUSH byte slice c of my shard into every rank's workspace, nearest consumer
// first (rank-1 starts with my rows right after its own; at any moment every rank pushes to a different peer,
// so each NVLink port carries one stream per direction).
//
// Mechanism chosen from measurements on B200 (profiles/p2p_mechanisms_2xB200.json and the intra-kernel
// profiles in profiles/): coalesced 16-byte generic stores from all 256 threads move ~42 GB/s per SM and
// 16-32 SMs fill the port; the arrival flag needs a system-scope release AFTER the data (a relaxed flag store
// following cp.async.bulk completion was observed to overtake the data), and that fence is expensive while
// the SM has NVLink writes in flight -- so it is issued once per (CTA, destination), after a whole slice.
// -------------------------------------------------------------------------------------------------
// 8-bit kinds: the scales that belong to rows [r0, r1) of my shard, stored by all threads of a comm CTA into rank d's workspace
// half par, BEFORE the release fence that publishes the rows (so the rows' flag covers them; there are no extra flags):
//  * per-row activation scales (int8 / e4m3; with_rows): scale_a[r] -> ag_scale_ws[par][me * Ms + r].  A per-tensor scale was
//    expanded to my rows by the caller, so every source's rows carry their own rank's scale.
//  * MXFP8: the 512-byte chunks of k-blocks [kb0, kb1) of every 128-row block whose FIRST row lies in [r0, r1).  That block's
//    first row is pushed by this CTA, so a consumer waiting for the first row's flag (ag_wait_rows / ag_wait_kslice) has the chunk.
TD_DEVICE void ag_push_scales(const Params& p, uint32_t par, int d, int r0, int r1, int kb0, int kb1, bool with_rows) {
  const int me = p.symm.rank, Ms = p.ag_rows_per_rank;
  if (with_rows && p.ag_scale_ws != nullptr) {
    const size_t rows_buf = p.ag_ws_buf_bytes / (static_cast<size_t>(p.K) * p.ag_esz);
    float* dst = symm_at(p.symm, p.ag_scale_ws + par * rows_buf + static_cast<size_t>(me) * Ms, d);
    for (int r = r0 + static_cast<int>(threadIdx.x); r < r1; r += kThreads) dst[r] = p.scale_a[r];
  }
  if (p.ag_sf_ws != nullptr) {
    const int b0 = (r0 + BM - 1) / BM, b1 = (r1 + BM - 1) / BM, nkb = kb1 - kb0;
    constexpr int kPieces = kSFChunk / 16;
    const int n = max(0, b1 - b0) * max(0, nkb) * kPieces;
    char* dst = symm_at(p.symm, p.ag_sf_ws + (static_cast<size_t>(par) * p.ag_sf_buf_chunks + static_cast<size_t>(me) * (Ms / BM) * p.num_k) * kSFChunk, d);
    for (int i = threadIdx.x; i < n; i += kThreads) {
      const int c = i / kPieces;
      const size_t off = (static_cast<size_t>(b0 + c / nkb) * p.num_k + kb0 + c % nkb) * kSFChunk + (i % kPieces) * 16;
      ptx::st_na_v4(dst + off, ptx::ld_nc_v4(p.ag_sf_local + off));
    }
  }
}

TD_DEVICE void ag_comm_cta(const Params& p, uint32_t ph, int comm_idx) {
  const int W = p.symm.world, me = p.symm.rank, Ms = p.ag_rows_per_rank;
  const size_t row_bytes = static_cast<size_t>(p.K) * p.ag_esz;
  const size_t shard_bytes = static_cast<size_t>(Ms) * row_bytes;
  const size_t slice = ag_slice_bytes(shard_bytes, p.ag_nslices);
  char* ws = p.ag_ws + (ph & 1u) * p.ag_ws_buf_bytes;
  const size_t shard_off = static_cast<size_t>(me) * Ms * row_bytes;
  const char* src0 = p.ag_copy_local ? reinterpret_cast<const char*>(p.ag_a_local) : ws + shard_off;
  uint32_t* flag_base = p.ag_flags + (ph & 1u) * W * kAGMaxSlices + me * kAGMaxSlices;
  const int pslot = static_cast<int>(blockIdx.x) * 8;
  // ag_nslices = n_comm * nsub: with few destinations (TP2 / TP4) a CTA cuts its share into nsub sub-slices that are
  // interleaved over the shard (sub-slice j of all CTAs = the j-th 1/nsub of the rows), each published separately, so
  // the consumer's first remote tiles become ready after 1/nsub of the transfer instead of at its end
  const int nsub = max(1, p.ag_nslices / max(1, p.n_comm_ctas));
  if (p.ag_kslices > 0) {
    // K-sliced transports.  ag_multicast = 1 (NVLS): one multimem.st per 16 bytes reaches every rank's workspace; egress is the shard
    // itself, not (world - 1) copies of it, so a handful of CTAs is enough.  The shard travels K slice by K slice
    // (all rows of columns [j * seg, (j + 1) * seg)), so on the consumer EVERY tile starts after 1 / ag_kslices of the
    // transfer and its mainloop follows the arrival: the tail after the last byte is one K slice of MMAs + the epilogue.
    // ag_multicast = 0 (P2P): the same slices are stored to every peer's workspace with unicast 16-byte stores -- the rows are
    // READ once and written W-1 times, and there is ONE release fence per (CTA, slice) for all destinations (a fence after
    // NVLink stores costs ~7 us of latency: the per-destination fences of the row-sliced path cost 7 x that).  Measured on
    // 8xB200: multimem.st tops out near 380 GB/s of ingress per GPU, unicast stores reach the link rate.
    char* ws_mc = p.ag_multicast ? symm_mc(p.symm, ws) + shard_off : nullptr;
    const int n_c = p.ag_ctas_per_group, n_groups = p.n_comm_ctas / n_c;
    const int grp = comm_idx / n_c, cta = comm_idx % n_c;
    const int r0 = cta * p.ag_rows_per_cta, r1 = min(Ms, r0 + p.ag_rows_per_cta);
    for (int j = grp; j < p.ag_kslices; j += n_groups) {
      const size_t col0 = static_cast<size_t>(p.ag_slice_kb[j]) * 128;
      const int seg16 = static_cast<int>((min(row_bytes, static_cast<size_t>(p.ag_slice_kb[j + 1]) * 128) - col0) >> 4);
      const int n = max(0, r1 - r0) * seg16;
      if (threadIdx.x == 0) prof_record(p.prof, pslot, 1, true);
      // 16 independent 16-byte loads per thread before the first store (the copy loop is bound by the latency of its reads)
      constexpr int U = 16;
      auto off_of = [&](int i) { return static_cast<size_t>(r0 + i / seg16) * row_bytes + col0 + static_cast<size_t>(i % seg16) * 16; };
      for (int i0 = threadIdx.x; i0 < n; i0 += U * kThreads) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int i = i0 + u * kThreads;
          if (i < n) v[u] = ptx::ld_nc_v4(src0 + off_of(i));
        }
        if (p.ag_multicast) {
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kThreads;
            if (i < n) ptx::multimem_st_v4(ws_mc + off_of(i), v[u]);
          }
        } else {
          for (int q = 1; q < W; ++q) {          // every rank starts with a different peer: all links busy at any instant
            char* dst = symm_at(p.symm, ws, (me + q) % W) + shard_off;
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const int i = i0 + u * kThreads;
              if (i < n) ptx::st_na_v4(dst + off_of(i), v[u]);
            }
          }
        }
      }
      if (p.ag_scale_ws != nullptr || p.ag_sf_ws != nullptr)   // scales of my rows with slice 0, MXFP8 chunks of slice j's k-blocks
        for (int d = (p.ag_multicast || !p.ag_local_direct) ? 0 : 1; d < W; ++d)
          ag_push_scales(p, ph & 1u, (me + d) % W, r0, r1, p.ag_slice_kb[j], p.ag_slice_kb[j + 1], j == 0);
      __syncthreads();
      if (threadIdx.x == 0) {
        prof_record(p.prof, pslot, 1, false);
        prof_record(p.prof, pslot, 6, true);
        ptx::fence_acq_rel_sys();
        for (int d = (p.ag_multicast || !p.ag_local_direct) ? 0 : 1; d < W; ++d) ptx::st_relaxed_sys(symm_at(p.symm, flag_base + j * n_c + cta, (me + d) % W), ph);
        prof_record(p.prof, pslot, 6, false);
      }
    }
    return;
  }
  for (int dist = (p.ag_copy_local && !p.ag_local_direct) ? 0 : 1; dist < W; ++dist) {
    const int d = (me - dist + W) % W;
    // ag_copy_local == 2: all-to-all flavour -- a_local is [world, rows_per_rank, K] and block d goes to rank d
    const size_t a2a_off = (p.ag_copy_local == 2) ? static_cast<size_t>(d) * shard_bytes : 0;
    for (int j = 0; j < nsub; ++j) {
      const int sidx = j * p.n_comm_ctas + comm_idx;
      const size_t b0 = min(shard_bytes, slice * sidx), b1 = min(shard_bytes, b0 + slice);
      if (threadIdx.x == 0) prof_record(p.prof, pslot, 1, true);
      if (b1 > b0) copy16_strided_deep(symm_at(p.symm, ws, d) + shard_off + b0, src0 + a2a_off + b0, b1 - b0, threadIdx.x, kThreads);
      if (p.ag_scale_ws != nullptr || p.ag_sf_ws != nullptr)   // rows whose first byte is in this slice
        ag_push_scales(p, ph & 1u, d, static_cast<int>((b0 + row_bytes - 1) / row_bytes), static_cast<int>((b1 + row_bytes - 1) / row_bytes),
                       0, p.num_k, true);
      __syncthreads();
      if (threadIdx.x == 0) {
        prof_record(p.prof, pslot, 1, false);
        prof_record(p.prof, pslot, 6, true);
        ptx::fence_acq_rel_sys();
        ptx::st_relaxed_sys(symm_at(p.symm, flag_base + sidx, d), ph);
        prof_record(p.prof, pslot, 6, false);
      }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// AR consumer side (comm CTA c): tiles c, c + n_comm, ... in the order the GEMM produces them.  A tile is
// complete when all W ranks have published flag[par][tile][rank] = phase; the reduction is one
// multimem.ld_reduce per 16 bytes (the switch adds the W staging copies) or W peer loads without NVLS.
// -------------------------------------------------------------------------------------------------
template <int kCtaGroup, int BN>
TD_DEVICE void ar_comm_cta(const Params& p, uint32_t ph, int comm_idx) {
  constexpr int TM = BM * kCtaGroup;
  const int W = p.symm.world;
  const int total_tiles = p.num_m * p.num_n;
  char* stage = p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes;
  const uint32_t* flags = p.rs_flags + static_cast<size_t>(ph & 1u) * p.rs_flag_tiles * W;
  constexpr int kChunksPerRow = BN / 8;
  for (int t = comm_idx; t < total_tiles; t += p.n_comm_ctas) {
    int m_tile, n_tile;
    tile_coords(p, t, m_tile, n_tile);
    if (static_cast<int>(threadIdx.x) < W * kCtaGroup) {      // one waiter per (row half, source rank)
      const int half = static_cast<int>(threadIdx.x) / W, src = static_cast<int>(threadIdx.x) % W;
      wait_ge<true>(flags + static_cast<size_t>((m_tile * kCtaGroup + half) * p.num_n + n_tile) * W + src, ph);
    }
    __syncthreads();
    const int row0 = m_tile * TM, col0 = n_tile * BN;
    if (p.symm.mc_base) {
      // NVLS: 4 independent multimem.ld_reduce per thread in flight (the switch round trip is ~2 us)
      constexpr int U = 4;
      for (int i0 = threadIdx.x; i0 < TM * kChunksPerRow; i0 += U * kThreads) {
        uint4 v[U]; char* dst[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int i = i0 + u * kThreads;
          const int r = row0 + i / kChunksPerRow, c = col0 + (i % kChunksPerRow) * 8;
          dst[u] = nullptr;
          if (i < TM * kChunksPerRow && r < p.M && c < p.N) {
            char* src = stage + (static_cast<size_t>(r) * p.N + c) * 2;
            v[u] = p.in_is_bf16 ? ptx::multimem_ld_reduce_bf16x8(symm_mc(p.symm, src)) : ptx::multimem_ld_reduce_f16x8(symm_mc(p.symm, src));
            dst[u] = reinterpret_cast<char*>(p.rs_out) + (static_cast<size_t>(r) * p.rs_ldo + c) * 2;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (dst[u]) ptx::st_v4(dst[u], v[u]);
      }
    } else {
      for (int i = threadIdx.x; i < TM * kChunksPerRow; i += kThreads) {
        const int r = row0 + i / kChunksPerRow, c = col0 + (i % kChunksPerRow) * 8;
        if (r >= p.M || c >= p.N) continue;
        char* src = stage + (static_cast<size_t>(r) * p.N + c) * 2;
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int s = 0; s < W; ++s) {
          const uint4 x = ptx::ld_relaxed_sys_v4(symm_at(p.symm, src, (p.symm.rank + s) % W));
          const uint32_t w4[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (p.in_is_bf16) { acc[2 * e] += ptx::bf16_lo(w4[e]); acc[2 * e + 1] += ptx::bf16_hi(w4[e]); }
            else { const __half2 hh = *reinterpret_cast<const __half2*>(&w4[e]); acc[2 * e] += __low2float(hh); acc[2 * e + 1] += __high2float(hh); }
          }
        }
        uint4 v;
        if (p.in_is_bf16) { v.x = ptx::pack_bf16x2(acc[0], acc[1]); v.y = ptx::pack_bf16x2(acc[2], acc[3]); v.z = ptx::pack_bf16x2(acc[4], acc[5]); v.w = ptx::pack_bf16x2(acc[6], acc[7]); }
        else { v.x = ptx::pack_f16x2(acc[0], acc[1]); v.y = ptx::pack_f16x2(acc[2], acc[3]); v.z = ptx::pack_f16x2(acc[4], acc[5]); v.w = ptx::pack_f16x2(acc[6], acc[7]); }
        ptx::st_v4(reinterpret_cast<char*>(p.rs_out) + (static_cast<size_t>(r) * p.rs_ldo + c) * 2, v);
      }
    }
    __syncthreads();
  }
}

// -------------------------------------------------------------------------------------------------
// MoE reduce-RS comm CTA ci: per n tile c (= chunk of BN output columns)
//   (1) wait until every valid m tile of chunk c has been scattered to y (= p.C, [T * topk, N], rows already weighted)
//   (2) sum the top-k rows of my token slice into my symmetric partial part[t][chunk]
//   (3) release-flag every rank: flag[par][c][me][ci] = phase
//   (4) one chunk later: wait for the W ranks' flags of the slices that cover the rows I pull and reduce them through the
//       NVSwitch (multimem.ld_reduce, fp32 accumulation) -- or W peer loads without NVLS -- into the output
// Reduce-scatter: rank r pulls tokens [r * T / W, (r + 1) * T / W); all-reduce: every rank pulls every token.
// -------------------------------------------------------------------------------------------------
TD_DEVICE void acc_16bit(float (&acc)[8], const uint4& x, bool bf16) {
  const uint32_t w4[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (bf16) { acc[2 * e] += ptx::bf16_lo(w4[e]); acc[2 * e + 1] += ptx::bf16_hi(w4[e]); }
    else { const __half2 hh = *reinterpret_cast<const __half2*>(&w4[e]); acc[2 * e] += __low2float(hh); acc[2 * e + 1] += __high2float(hh); }
  }
}
TD_DEVICE uint4 pack_16bit(const float (&acc)[8], bool bf16) {
  uint4 v;
  if (bf16) { v.x = ptx::pack_bf16x2(acc[0], acc[1]); v.y = ptx::pack_bf16x2(acc[2], acc[3]); v.z = ptx::pack_bf16x2(acc[4], acc[5]); v.w = ptx::pack_bf16x2(acc[6], acc[7]); }
  else { v.x = ptx::pack_f16x2(acc[0], acc[1]); v.y = ptx::pack_f16x2(acc[2], acc[3]); v.z = ptx::pack_f16x2(acc[4], acc[5]); v.w = ptx::pack_f16x2(acc[6], acc[7]); }
  return v;
}

// MoE reduce-RS, every CTA at kernel start: zero my slice of this call's partial buffer (the epilogues ADD into it), then count
// myself in.  part[par] was last read by the peers' pulls of call i-2, which all ended before any peer flagged call i-1 -- and I
// only finished call i-1 after seeing those flags -- so it is free.  Epilogues wait for all CTAs before their first reduction.
TD_DEVICE void moe_rs_zero_part(const Params& p, uint32_t ph) {
  const uint32_t par = ph & 1u;
  uint4* part = reinterpret_cast<uint4*>(p.rs_stage + par * p.rs_stage_buf_bytes);
  const size_t n16 = static_cast<size_t>(p.mrs_T) * p.N * 2 / 16;
  const size_t per = (n16 + gridDim.x - 1) / gridDim.x;
  const size_t i0 = min(n16, per * blockIdx.x), i1 = min(n16, i0 + per);
  for (size_t i = i0 + threadIdx.x; i < i1; i += kThreads) part[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  if (threadIdx.x == 0) { __threadfence(); ptx::red_release_gpu_add(p.mrs_counter + par * (p.mrs_n_chunks + 1) + p.mrs_n_chunks, 1u); }
}

// MoE reduce-RS comm CTA ci: for every column chunk (in the order the GEMM finishes them) wait for the W ranks' "chunk done"
// flags and reduce the rows I pull through the NVSwitch (multimem.ld_reduce, fp32 accumulation; W peer loads without NVLS).
// Reduce-scatter: rank r pulls tokens [r * T / W, (r + 1) * T / W); all-reduce: every rank pulls every token.
template <int BN>
TD_DEVICE void moe_rs_comm_cta(const Params& p, uint32_t ph, int ci) {
  const int W = p.symm.world, me = p.symm.rank, nc = p.n_comm_ctas, T = p.mrs_T, N = p.N;
  const int n_chunks = p.mrs_n_chunks;
  const uint32_t par = ph & 1u;
  const bool bf16 = p.in_is_bf16 != 0;
  if (ci == 0)
    for (int i = threadIdx.x; i <= n_chunks; i += kThreads) p.mrs_counter[(par ^ 1u) * (n_chunks + 1) + i] = 0u;   // the NEXT call's counters
  char* part = p.rs_stage + par * p.rs_stage_buf_bytes;
  const uint32_t* flags = p.rs_flags + static_cast<size_t>(par) * n_chunks * W;
  int r0, r1, out_row0;
  if (p.mrs_allreduce) { const int per = (T + nc - 1) / nc; r0 = min(T, ci * per); r1 = min(T, r0 + per); out_row0 = 0; }
  else {
    const int Tr = T / W, rows_per = (Tr + nc - 1) / nc;
    r0 = me * Tr + min(Tr, ci * rows_per); r1 = me * Tr + min(Tr, (ci + 1) * rows_per); out_row0 = me * Tr;
  }
  constexpr int U = 8;          // multimem.ld_reduce round trips (~3 us through the switch) in flight per thread
  for (int c = 0; c < n_chunks; ++c) {
    if (static_cast<int>(threadIdx.x) < W) wait_ge<true>(flags + static_cast<size_t>(c) * W + threadIdx.x, ph);
    __syncthreads();
    const int col0 = p.mrs_chunk_start[c] * BN, col1 = min(N, p.mrs_chunk_start[c + 1] * BN);
    const int cpr = (col1 - col0) / 8;                   // 16-byte pieces per row of this chunk
    const int items = (r1 - r0) * cpr;
    for (int i0 = threadIdx.x; i0 < items; i0 += U * kThreads) {
      uint4 v[U];
      if (p.symm.mc_base) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int i = i0 + u * kThreads;
          if (i < items) {
            char* src = part + (static_cast<size_t>(r0 + i / cpr) * N + col0 + (i % cpr) * 8) * 2;
            v[u] = bf16 ? ptx::multimem_ld_reduce_bf16x8(symm_mc(p.symm, src)) : ptx::multimem_ld_reduce_f16x8(symm_mc(p.symm, src));
          }
        }
      } else {
        float acc[U][8];
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[u][e] = 0.f;
        }
        for (int s = 0; s < W; ++s) {
          uint4 x[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kThreads;
            if (i < items) x[u] = ptx::ld_relaxed_sys_v4(symm_at(p.symm, part + (static_cast<size_t>(r0 + i / cpr) * N + col0 + (i % cpr) * 8) * 2, (me + s) % W));
          }
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (i0 + u * kThreads < items) acc_16bit(acc[u], x[u], bf16);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = pack_16bit(acc[u], bf16);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * kThreads;
        if (i < items)
          ptx::st_v4(reinterpret_cast<char*>(p.rs_out) + (static_cast<size_t>(r0 + i / cpr - out_row0) * p.rs_ldo + col0 + (i % cpr) * 8) * 2, v[u]);
      }
    }
    __syncthreads();
  }
}

// -------------------------------------------------------------------------------------------------
// Mega-EP dispatch comm CTA: CTA ci serves destination d = (me + ci / cpd) % W (every rank starts with itself, then a different
// peer each) and, expert by expert (local expert e of d = global expert d * epr + e), stores its share of my rows routed to
// that expert -- one warp per row, 16 B vectors, 4 loads in flight per lane -- into rows [dest_off[g], ...) of d's A matrix
// plus the 4-byte return address; then ONE release fence and the flag of (e, me, my sub-index) on d.  Experts are sent in
// the order the destination's GEMM consumes them.
// -------------------------------------------------------------------------------------------------
TD_DEVICE void epd_comm_cta(const Params& p, uint32_t ph, int ci) {
  const int W = p.symm.world, me = p.symm.rank, cpd = p.epd_cpd;
  const int d = (me + ci / cpd) % W, sub = ci % cpd;
  const uint32_t par = ph & 1u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpc = kThreads / 32;
  const size_t row_bytes = static_cast<size_t>(p.K) * 2;
  const int vecs = static_cast<int>(row_bytes >> 4);
  char* rx = symm_at(p.symm, p.ag_ws + par * p.ag_ws_buf_bytes, d);
  uint32_t* meta = symm_at(p.symm, p.epd_meta + static_cast<size_t>(par) * p.epd_rows_cap, d);
  for (int e = 0; e < p.epd_epr; ++e) {
    const int g = d * p.epd_epr + e;
    const int base = p.epd_send_off[g], n = p.epd_send_off[g + 1] - base, drow0 = p.epd_dest_off[g];
    for (int i = sub * wpc + warp; i < n; i += cpd * wpc) {
      const int drow = drow0 + i;
      if (drow >= p.epd_rows_cap) continue;                       // over capacity: dropped (the host sized the buffers)
      const int pair = p.epd_send_ids[base + i];
      const uint4* src = reinterpret_cast<const uint4*>(p.epd_x + static_cast<size_t>(pair / p.epd_topk) * row_bytes);
      uint4* dst = reinterpret_cast<uint4*>(rx + static_cast<size_t>(drow) * row_bytes);
      int v = lane;
      for (; v + 96 < vecs; v += 128) {
        const uint4 a0 = ptx::ld_nc_v4(src + v), a1 = ptx::ld_nc_v4(src + v + 32), a2 = ptx::ld_nc_v4(src + v + 64), a3 = ptx::ld_nc_v4(src + v + 96);
        ptx::st_na_v4(dst + v, a0); ptx::st_na_v4(dst + v + 32, a1); ptx::st_na_v4(dst + v + 64, a2); ptx::st_na_v4(dst + v + 96, a3);
      }
      for (; v < vecs; v += 32) ptx::st_na_v4(dst + v, ptx::ld_nc_v4(src + v));
      if (lane == 0) meta[drow] = (static_cast<uint32_t>(me) << 24) | static_cast<uint32_t>(pair);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      ptx::fence_acq_rel_sys();
      uint32_t* f = p.epd_flags + ((static_cast<size_t>(par) * p.epd_epr + e) * W + me) * cpd + sub;
      ptx::st_relaxed_sys(symm_at(p.symm, f, d), ph);
    }
  }
}
// consumer: all rows of local expert e (from every source, every comm CTA) have landed in my A matrix
TD_DEVICE void epd_wait_expert(const Params& p, uint32_t ph, int e) {
  const int n = p.symm.world * p.epd_cpd;
  const uint32_t* f = p.epd_flags + (static_cast<size_t>(ph & 1u) * p.epd_epr + e) * n;
  for (int i = 0; i < n; ++i) wait_ge<true>(f + i, ph);
  ptx::fence_proxy_async();
}

// -------------------------------------------------------------------------------------------------
// the kernel
// -------------------------------------------------------------------------------------------------
template <int kMode, int BN, int kStages, int kCtaGroup, bool kFP8 = false, int kAccStages = 2>
__global__ void __launch_bounds__(kThreads, 1) gemm_kernel(const __grid_constant__ Params p) {
  using L = SmemLayout<BN, kStages, kCtaGroup, 0, kFP8>;
  const int kBKElems = kFP8 ? 128 : p.bk_elems;         // K elements per 128-byte smem row (128 for every 8-bit kind)
  constexpr int kSFCols = 4 + 4 * ((BN + 127) / 128);    // TMEM columns of scale factors per pipeline stage (A + B)
  constexpr int kSFBase = kAccStages * BN;               // scale factors live after the accumulator stage(s)
  static_assert(!kFP8 || (kAccStages * BN + kStages * kSFCols <= 512), "TMEM: accumulators + scale-factor ring exceed 512 columns");
  constexpr int TM = BM * kCtaGroup;                     // rows of C per cluster tile
  constexpr int kTmemCols = kFP8 ? 512 : tmem_cols_for(BN);
  constexpr int kNumCBlocks = (BN + kCBlockCols - 1) / kCBlockCols;
  constexpr int kColsPerBlock = BN < kCBlockCols ? BN : kCBlockCols;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (kCtaGroup == 2) ? ptx::cluster_ctarank() : 0u;
  const bool is_leader = cta_rank == 0;
  const uint32_t ph = (kMode == kPlain) ? 0u : (p.phase[0] + 1u);
  const int cbuf = p.c_phase ? static_cast<int>((p.c_phase[0] + 1u) & 1u) : 0;

  const int n_gemm_ctas = static_cast<int>(gridDim.x) - p.n_comm_ctas;
  const bool is_comm = static_cast<int>(blockIdx.x) >= n_gemm_ctas;

  if constexpr (kMode == kMoeRS) moe_rs_zero_part(p, ph);
  if (is_comm) {
    // dedicated comm CTA (fills the SMs the GEMM has no tiles for): deep ring, one driving thread
    if constexpr (kMode == kAG) {
      ag_comm_cta(p, ph, static_cast<int>(blockIdx.x) - n_gemm_ctas);
    }
    if constexpr (kMode == kAR) {
      ar_comm_cta<kCtaGroup, BN>(p, ph, static_cast<int>(blockIdx.x) - n_gemm_ctas);
    }
    if constexpr (kMode == kMoeRS) {
      moe_rs_comm_cta<BN>(p, ph, static_cast<int>(blockIdx.x) - n_gemm_ctas);
    }
    if constexpr (kMode == kEPD) {
      epd_comm_cta(p, ph, static_cast<int>(blockIdx.x) - n_gemm_ctas);
    }
  } else {
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    if (warp == 0 && lane == 0) {
      ptx::prefetch_tensormap(&p.tmap_a);
      ptx::prefetch_tensormap(&p.tmap_b);
      if (p.use_tma_store) ptx::prefetch_tensormap(&p.tmap_c);
    }
    if (warp == 1 && lane == 0) {
      for (int i = 0; i < kStages; ++i) {
        ptx::mbar_init(full_bar + i, kCtaGroup);      // one producer arrival per CTA of the pair (+ tx bytes)
        ptx::mbar_init(empty_bar + i, 1);             // one tcgen05.commit
      }
      for (int i = 0; i < 2; ++i) {
        ptx::mbar_init(tmem_full + i, 1);                       // one tcgen05.commit
        ptx::mbar_init(tmem_empty + i, 4 * kCtaGroup);          // one arrival per epilogue warp of the pair
      }
      ptx::fence_barrier_init();
    }
    if (warp == 2) {
      ptx::tmem_alloc<kCtaGroup>(tmem_ptr_smem, kTmemCols);
      ptx::tmem_relinquish<kCtaGroup>();
    }
    ptx::tc_fence_before();
    if constexpr (kCtaGroup == 2) ptx::cluster_sync(); else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    const int n_workers = n_gemm_ctas / kCtaGroup;                 // clusters that run GEMM tiles
    const int worker = static_cast<int>(blockIdx.x) / kCtaGroup;
    const int total_tiles = p.num_m * p.num_n;

    if (warp == 0 && p.a_gather != nullptr) {
      // ================================ TMA producer, gathered A (whole warp) ================================
      // lane l owns rows 4l..4l+3 of the 128-row tile: one tile::gather4 per k-block per lane, B by lane 0
      if constexpr (kCtaGroup == 1 && !kFP8) {
        int stage = 0; uint32_t phase = 0;
        for (int u = worker; u < p.total_units; u += n_workers) {
          const Unit un = get_unit(p, u);
          int m_tile, n_tile;
          tile_coords(p, un.tile, m_tile, n_tile);
          int expert = 0;
          if (p.tile_expert) { expert = p.tile_expert[m_tile]; if (expert < 0) continue; }
          const int row0 = m_tile * TM;
          const int brow0 = expert * p.expert_rows + n_tile * BN;
          int4 id = make_int4(-1, -1, -1, -1);
          if (row0 + 4 * lane < p.M) id = *reinterpret_cast<const int4*>(p.a_gather + row0 + 4 * lane);
          const int dv = p.a_gather_div, pad = p.a_gather_pad;
          const int r0 = (id.x == pad || id.x < 0) ? -1 : id.x / dv, r1 = (id.y == pad || id.y < 0) ? -1 : id.y / dv;
          int r2 = (id.z == pad || id.z < 0) ? -1 : id.z / dv, r3 = (id.w == pad || id.w < 0) ? -1 : id.w / dv;
          int r0m = r0, r1m = r1;
          if constexpr (kMode == kAG) {
            // fused AllGather + grouped GEMM: the rows live in the all-gather workspace; each lane waits for the byte
            // slices (source rank, comm CTA) that carry ITS four rows, then the rows are gathered by TMA
            const int rr[4] = {r0, r1, r2, r3};
            const int Ms = p.ag_rows_per_rank;
            const size_t row_bytes = static_cast<size_t>(p.K) * p.ag_esz;
            const size_t slice = ag_slice_bytes(static_cast<size_t>(Ms) * row_bytes, p.ag_nslices);
            const uint32_t* flags = p.ag_flags + (ph & 1u) * p.symm.world * kAGMaxSlices;
            if (!p.ag_skip_wait) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                if (rr[q] < 0) continue;
                const int s = rr[q] / Ms;
                if (s == p.symm.rank && !p.ag_copy_local) continue;
                const size_t b0 = static_cast<size_t>(rr[q] - s * Ms) * row_bytes;
                for (int c = static_cast<int>(b0 / slice); c <= static_cast<int>((b0 + row_bytes - 1) / slice); ++c)
                  wait_ge<true>(flags + s * kAGMaxSlices + c, ph);
              }
              ptx::fence_proxy_async();
            }
            const int par_rows = static_cast<int>((ph & 1u) * (p.ag_ws_buf_bytes / row_bytes));   // parity half of the workspace
            if (r0m >= 0) r0m += par_rows;
            if (r1m >= 0) r1m += par_rows;
            if (r2 >= 0) r2 += par_rows;
            if (r3 >= 0) r3 += par_rows;
          }
          __syncwarp();
          for (int kb = un.kb0; kb < un.kb1; ++kb) {
            if (lane == 0) {
              ptx::mbar_wait(empty_bar + stage, phase ^ 1u);
              ptx::mbar_arrive_expect_tx(full_bar + stage, L::kTxBytes);
            }
            __syncwarp();
            uint8_t* sa = smem + stage * L::kStageBytes;
            ptx::tma_gather4_2d(&p.tmap_ag, full_bar + stage, sa + lane * 512, kb * kBKElems, r0m, r1m, r2, r3);
            if (lane == 0) ptx::tma_load_2d(&p.tmap_b, full_bar + stage, sa + L::kABytes, kb * kBKElems, brow0, ptx::kEvictLast);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
      __syncwarp();
    } else if (warp == 0) {
      // ================================ TMA producer ================================
      if (lane == 0) {
        int stage = 0; uint32_t phase = 0;
        int epd_seen = -1;
        (void)epd_seen;
        for (int u = worker; u < p.total_units; u += n_workers) {
          const Unit un = get_unit(p, u);
          if (un.kb1 <= un.kb0) continue;                    // empty K segment (the output was zero-filled by the caller)
          int m_tile, n_tile;
          tile_coords(p, un.tile, m_tile, n_tile);
          int expert = 0;
          if (p.tile_expert) { expert = p.tile_expert[m_tile]; if (expert < 0) continue; }
          const int row0 = m_tile * TM + static_cast<int>(cta_rank) * BM;       // my 128 rows of A
          const int brow0 = expert * p.expert_rows + n_tile * BN + static_cast<int>(cta_rank) * (BN / kCtaGroup);
          if constexpr (kMode == kAG) {
            prof_record(p.prof, static_cast<int>(blockIdx.x) * 8, 3, true);
            if (!p.ag_skip_wait && !p.ag_kslices && row0 < p.M) ag_wait_rows(p, ph, row0, min(p.M, row0 + BM));
            prof_record(p.prof, static_cast<int>(blockIdx.x) * 8, 3, false);
          }
          const int abuf = (kMode == kAG || kMode == kEPD) ? static_cast<int>(ph & 1u) : 0;
          if constexpr (kMode == kEPD) {
            if (!p.ag_skip_wait && expert != epd_seen) { epd_wait_expert(p, ph, expert); epd_seen = expert; }
          }
          // my own rows come straight from the caller's tensor (no local copy into the workspace)
          bool a_local = false; int lrow0 = 0;
          if constexpr (kMode == kAG) {
            if (p.ag_local_direct && row0 >= p.symm.rank * p.ag_rows_per_rank && row0 < (p.symm.rank + 1) * p.ag_rows_per_rank) {
              a_local = true;
              lrow0 = (p.ag_copy_local == 2) ? row0 : row0 - p.symm.rank * p.ag_rows_per_rank;
            }
          }
          // K-sliced all-gather: before the first k-block of every K slice, acquire that slice of my 128 rows
          const bool ks_wait = (kMode == kAG) && p.ag_kslices > 0 && !p.ag_skip_wait && !a_local && row0 < p.M;
          const int ks_src = ks_wait ? row0 / p.ag_rows_per_rank : 0;
          int ks_j = 0, ks_next = un.kb0;                 // current K slice and the k-block at which the next acquire is due
          for (int kb = un.kb0; kb < un.kb1; ++kb) {
            if constexpr (kMode == kAG) {
              if (ks_wait && kb == ks_next) {
                while (ks_j + 1 < p.ag_kslices && kb >= p.ag_slice_kb[ks_j + 1]) ++ks_j;
                ag_wait_kslice(p, ph, ks_src, row0 - ks_src * p.ag_rows_per_rank, ks_j);
                ks_next = p.ag_slice_kb[ks_j + 1];
              }
            }
            ptx::mbar_wait(empty_bar + stage, phase ^ 1u);
            uint8_t* sa = smem + stage * L::kStageBytes;
            uint8_t* sb = sa + L::kABytes;
            uint8_t* ssfa = sb + L::kBBytes;
            uint8_t* ssfb = ssfa + L::kSFABytes;
            if constexpr (kCtaGroup == 1) {
              ptx::mbar_arrive_expect_tx(full_bar + stage, L::kTxBytes);
              if (a_local) ptx::tma_load_2d(&p.tmap_al, full_bar + stage, sa, kb * kBKElems, lrow0);
              else ptx::tma_load_3d(&p.tmap_a, full_bar + stage, sa, kb * kBKElems, row0, abuf);
              ptx::tma_load_2d(&p.tmap_b, full_bar + stage, sb, kb * kBKElems, brow0, ptx::kEvictLast);
              if constexpr (kFP8) {
                if (a_local) ptx::tma_load_2d(&p.tmap_sfal, full_bar + stage, ssfa, 0, (lrow0 / 128) * p.num_k + kb);
                else ptx::tma_load_2d(&p.tmap_sfa, full_bar + stage, ssfa, 0, (row0 / 128) * p.num_k + kb + abuf * static_cast<int>(p.ag_sf_buf_chunks));
#pragma unroll
                for (int g = 0; g < (BN + 127) / 128; ++g)
                  ptx::tma_load_2d(&p.tmap_sfb, full_bar + stage, ssfb + g * kSFChunk, 0, ((n_tile * BN) / 128 + g) * p.num_k + kb);
              }
            } else {
              // both CTAs land their bytes on the LEADER's barrier; the leader expects both halves
              if (is_leader) ptx::mbar_arrive_expect_tx(full_bar + stage, 2 * L::kTxBytes);
              else ptx::mbar_arrive_cluster(full_bar + stage, 0);
              if (a_local) ptx::tma_load_2d_2sm(&p.tmap_al, full_bar + stage, sa, kb * kBKElems, lrow0);
              else ptx::tma_load_3d_2sm(&p.tmap_a, full_bar + stage, sa, kb * kBKElems, row0, abuf);
              ptx::tma_load_2d_2sm(&p.tmap_b, full_bar + stage, sb, kb * kBKElems, brow0, ptx::kEvictLast);
              if constexpr (kFP8) {
                if (a_local) ptx::tma_load_2d_2sm(&p.tmap_sfal, full_bar + stage, ssfa, 0, (lrow0 / 128) * p.num_k + kb);
                else ptx::tma_load_2d_2sm(&p.tmap_sfa, full_bar + stage, ssfa, 0, (row0 / 128) * p.num_k + kb + abuf * static_cast<int>(p.ag_sf_buf_chunks));
#pragma unroll
                for (int g = 0; g < (BN + 127) / 128; ++g)
                  ptx::tma_load_2d_2sm(&p.tmap_sfb, full_bar + stage, ssfb + g * kSFChunk, 0, ((n_tile * BN) / 128 + g) * p.num_k + kb);
              }
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ================================ MMA issuer (leader CTA, one thread) ================================
      if (is_leader && lane == 0) {
        const uint32_t idesc = p.in_kind == 1 ? ptx::make_idesc_i8(TM, BN)
                               : p.in_kind == 2 ? ptx::make_idesc(0u, 0u, TM, BN)
                                                : ptx::make_idesc(p.in_is_bf16 ? 1u : 0u, p.in_is_bf16 ? 1u : 0u, TM, BN);
        (void)idesc;
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int u = worker; u < p.total_units; u += n_workers) {
          const Unit un = get_unit(p, u);
          if (un.kb1 <= un.kb0) continue;
          if (p.tile_expert) {
            int m_tile, n_tile;
            tile_coords(p, un.tile, m_tile, n_tile);
            if (p.tile_expert[m_tile] < 0) continue;
          }
          ptx::mbar_wait(tmem_empty + acc, acc_phase ^ 1u);        // epilogue has drained this accumulator
          ptx::tc_fence_after();
          prof_record(p.prof, static_cast<int>(blockIdx.x) * 8 + 1, 4, true);
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
          // the k loop is instantiated once per operand kind (16-bit / int8 / e4m3): no per-MMA branch in the issuing thread
          auto k_loop = [&](auto kind_c) {
            constexpr int kKind = decltype(kind_c)::value;
            for (int kb = un.kb0; kb < un.kb1; ++kb) {
              ptx::mbar_wait(full_bar + stage, phase);
              ptx::tc_fence_after();
              const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
              const uint64_t adesc = ptx::make_smem_desc_k128(sa);
              const uint64_t bdesc = ptx::make_smem_desc_k128(sa + L::kABytes);
              if constexpr (!kFP8) {
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                  // advance 32 B (= 16 bf16) along K inside the 128-byte swizzle atom: +2 in the 16-byte address field
                  const uint32_t accf = (kb > un.kb0 || k != 0) ? 1u : 0u;
                  if constexpr (kKind == 0) ptx::mma_f16<kCtaGroup>(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, accf);
                  else if constexpr (kKind == 1) ptx::mma_i8<kCtaGroup>(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, accf);
                  else ptx::mma_f8f6f4<kCtaGroup>(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc, accf);
                }
              } else {
                // MXFP8: stage the UE8M0 scale factors of this k-block into TMEM (smem -> TMEM, 32 lanes x 16 B, replicated
                // to the four lane quadrants), then 4 block-scaled MMAs of K = 32; sf_id selects the byte of each 32-bit
                // scale word that belongs to the K-chunk.  tcgen05.cp and tcgen05.mma execute in issue order, so the
                // TMEM slot of this smem stage is free again by the time it is reused kStages k-blocks later.
                const uint32_t sf_tmem = tmem_base + static_cast<uint32_t>(kSFBase + stage * kSFCols);
                const uint32_t ssfa = sa + L::kABytes + L::kBBytes;
                ptx::tmem_cp_32x128b_warpx4<kCtaGroup>(sf_tmem, ptx::make_smem_desc_noswizzle(ssfa, 0, 128));
#pragma unroll
                for (int g = 0; g < (BN + 127) / 128; ++g)
                  ptx::tmem_cp_32x128b_warpx4<kCtaGroup>(sf_tmem + 4 + 4 * g,
                                                          ptx::make_smem_desc_noswizzle(ssfa + L::kSFABytes + g * kSFChunk, 0, 128));
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t idm = ptx::make_idesc_mx(0u, 0u, TM, BN, static_cast<uint32_t>(k), static_cast<uint32_t>(k));
                  ptx::mma_mxf8<kCtaGroup>(d_tmem, adesc + 2u * k, bdesc + 2u * k, idm, (kb > un.kb0 || k != 0) ? 1u : 0u, sf_tmem, sf_tmem + 4);
                }
              }
              if constexpr (kCtaGroup == 1) ptx::mma_commit(empty_bar + stage);
              else ptx::mma_commit_2sm(empty_bar + stage, 0b11);
              if (++stage == kStages) { stage = 0; phase ^= 1u; }
            }
          };
          if (kFP8 || p.in_kind == 0) k_loop(std::integral_constant<int, 0>{});
          else if (p.in_kind == 1) k_loop(std::integral_constant<int, 1>{});
          else k_loop(std::integral_constant<int, 2>{});
          if constexpr (kCtaGroup == 1) ptx::mma_commit(tmem_full + acc);
          else ptx::mma_commit_2sm(tmem_full + acc, 0b11);
          prof_record(p.prof, static_cast<int>(blockIdx.x) * 8 + 1, 4, false);
          if (++acc == kAccStages) { acc = 0; acc_phase ^= 1u; }
        }
      }
      __syncwarp();
    } else if (warp >= kEpiWarp0) {
      // ================================ epilogue ================================
      const int ew = warp - kEpiWarp0;               // == warp % 4 == TMEM lane quadrant
      const int et = threadIdx.x - kEpiWarp0 * 32;   // 0..127
      const int my_row = ew * 32 + lane;             // row of the 128-row CTA tile held by this thread
      uint8_t* smem_c = smem + L::kCOff;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t blk_iter = 0;                         // staging buffer = blk_iter & 1
      bool mrs_zero_seen = false;
      (void)mrs_zero_seen;
      for (int u = worker; u < p.total_units; u += n_workers) {
        const Unit un = get_unit(p, u);
        if (un.kb1 <= un.kb0) continue;
        int m_tile, n_tile;
        tile_coords(p, un.tile, m_tile, n_tile);
        if (p.tile_expert && p.tile_expert[m_tile] < 0) continue;
        const int row_base = m_tile * TM + static_cast<int>(cta_rank) * BM;   // global row of tile row 0
        const int cbuf_u = p.segk_off ? un.batch : cbuf;                      // output buffer of this unit
        const int col_base = n_tile * BN;

        if (un.part > 0) {
          // ---- split-K helper unit: park the fp32 accumulator of my K range in the workspace, raise the flag ----
          // layout per (32-column chunk, warp quadrant): [8 x 16-byte piece][32 lanes] -> every st.v4 / ld.v4 of a warp is
          // 512 contiguous bytes, and the reader (same row <-> thread mapping) adds piece by piece
          const size_t pidx = static_cast<size_t>(un.slot * (p.sk_parts - 1) + un.part - 1) * kCtaGroup + cta_rank;
          float* wsb = p.sk_ws + pidx * (BM * BN);
          ptx::mbar_wait(tmem_full + acc, acc_phase);
          ptx::tc_fence_after();
#pragma unroll 1
          for (int ch = 0; ch < BN / 32; ++ch) {
            uint32_t v[32];
            ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(acc * BN + ch * 32), v);
            ptx::tmem_ld_wait();
            float* dst = wsb + (ch * 4 + ew) * 1024 + lane * 4;
#pragma unroll
            for (int q = 0; q < 8; ++q) ptx::st_v4(dst + q * 128, make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (kCtaGroup == 1) ptx::mbar_arrive(tmem_empty + acc);
            else ptx::mbar_arrive_cluster(tmem_empty + acc, 0);
          }
          ptx::named_bar_sync(2, kEpiThreads);
          if (et == 0) { __threadfence(); ptx::st_release_gpu(p.sk_flags + pidx, 1u); }
          __syncwarp();
          if (++acc == kAccStages) { acc = 0; acc_phase ^= 1u; }
          continue;
        }
        const int sk_n = (un.slot >= 0) ? p.sk_parts - 1 : 0;     // partial accumulators to add (split-K part 0)
        float row_scale = 1.f;
        if (p.row_scale != nullptr && p.c_scatter != nullptr) {   // routing weight of the (token, k) pair this row is scattered to
          const int grow = row_base + my_row;
          const int id = grow < p.M ? p.c_scatter[grow] : -1;
          row_scale = (id >= 0 && id != p.a_gather_pad) ? p.row_scale[id] : 0.f;
        }

        // ---- RS ring bookkeeping for this tile ----
        int rs_step = 0; bool rs_final = false;
        const char* rs_in = nullptr;                 // running partial received from rank+1 (local memory)
        char* dst_base = reinterpret_cast<char*>(p.C) + cbuf_u * p.c_buf_stride_bytes;
        long long dst_ld = p.ldc;
        int dst_row_off = 0;                         // subtract from the global row for the destination
        bool f32_in = false, f32_out = false;        // fp32 ring staging (rs_fp32)
        if constexpr (kMode == kRS) {
          const int W = p.symm.world, me = p.symm.rank;
          const int owner = (m_tile * TM) / p.rs_rows_per_rank;
          rs_step = (owner - me - 1 + 2 * W) % W;
          rs_final = (rs_step == W - 1);
          char* stage_buf = p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes;
          if (rs_step > 0) {
            rs_in = stage_buf;
            if (et == 0 && !p.rs_skip_wait) wait_ge<true>(p.rs_flags + (ph & 1u) * total_tiles + m_tile * p.num_n + n_tile, ph);
            __syncwarp();
          }
          if (rs_final) {
            dst_base = reinterpret_cast<char*>(p.rs_out); dst_ld = p.rs_ldo; dst_row_off = owner * p.rs_rows_per_rank;
          } else {
            dst_base = symm_at(p.symm, stage_buf, (me - 1 + W) % W); dst_ld = p.N; dst_row_off = 0;
          }
          f32_in = p.rs_fp32 && rs_step > 0;
          f32_out = p.rs_fp32 && !rs_final;
        }

        int a2a_dst = 0;
        if constexpr (kMode == kAR) {
          if (p.a2a_cols_per_rank > 0) {   // scatter flavour: the tile's column block belongs to rank a2a_dst
            a2a_dst = col_base / p.a2a_cols_per_rank;
            dst_base = symm_at(p.symm, p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes, a2a_dst) -
                       static_cast<size_t>(a2a_dst) * p.a2a_cols_per_rank * 2;
            dst_ld = p.a2a_cols_per_rank; dst_row_off = -p.symm.rank * p.a2a_rows_per_src;
          } else {                         // partial tile -> my symmetric staging buffer (same coordinates as C)
            dst_base = p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes; dst_ld = p.N; dst_row_off = 0;
          }
        }

        if constexpr (kMode == kMoeRS) {
          // rows are ADDED to their token's row of my symmetric partial (top-k reduce at L2); first make sure it has been zeroed
          dst_base = p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes; dst_ld = p.N; dst_row_off = 0;
          if (!mrs_zero_seen) {
            if (et == 0) {
              const uint32_t* zc = p.mrs_counter + (ph & 1u) * (p.mrs_n_chunks + 1) + p.mrs_n_chunks;
              while (ptx::ld_acquire_gpu(zc) < gridDim.x) {}
            }
            ptx::named_bar_sync(2, kEpiThreads);
            mrs_zero_seen = true;
          }
        }
        ptx::mbar_wait(tmem_full + acc, acc_phase);
        ptx::tc_fence_after();
        if (lane == 0) prof_record(p.prof, static_cast<int>(blockIdx.x) * 8 + warp, 5, true);
        if (sk_n > 0) {     // the helper units of this tile run concurrently on other clusters: wait for their partials
          if (et < sk_n) {
            const uint32_t* f = p.sk_flags + static_cast<size_t>(un.slot * (p.sk_parts - 1) + et) * kCtaGroup + cta_rank;
            while (ptx::ld_acquire_gpu(f) == 0u) {}
          }
          ptx::named_bar_sync(2, kEpiThreads);
        } else if constexpr (kMode == kRS) { if (rs_step > 0) ptx::named_bar_sync(2, kEpiThreads); }  // flag acquired by et==0
        // kAG, int8 / e4m3: the per-row scale of a gathered row.  Own rows read the caller's scale_a (never written during the
        // launch).  A peer's scale was stored into ag_scale_ws by the comm CTA that pushed the row, before the release fence of
        // that row's flag (ag_push_scales).  The TMA producer acquired the flag, but the only path from that acquire to these
        // plain loads runs through TMA completion, tcgen05.mma and tcgen05.commit, which the memory model does not spell out as
        // a release / acquire chain.  So one thread re-acquires the flags of the tile's rows (already raised: one load each)
        // and the named barrier orders the other epilogue threads' loads after that acquire, as for the RS partials above.
        float ag_row_sa = 1.f;
        if constexpr (kMode == kAG) {
          if (p.ag_scale_ws != nullptr && row_base < p.M) {
            const int Ms = p.ag_rows_per_rank, s0 = row_base / Ms;
            if (!p.ag_skip_wait) {
              if (et == 0) {
                if (!p.ag_kslices) ag_wait_rows(p, ph, row_base, min(p.M, row_base + BM));
                else if (s0 != p.symm.rank) ag_wait_kslice(p, ph, s0, row_base - s0 * Ms, 0);
              }
              ptx::named_bar_sync(2, kEpiThreads);
            }
            const int grow = row_base + my_row;
            if (grow < p.M) {
              const int s = grow / Ms;
              const size_t rows_buf = p.ag_ws_buf_bytes / (static_cast<size_t>(p.K) * p.ag_esz);
              ag_row_sa = s == p.symm.rank ? p.scale_a[grow - s * Ms] : p.ag_scale_ws[(ph & 1u) * rows_buf + grow];
            }
          }
        }

#pragma unroll 1
        for (int cb = 0; cb < kNumCBlocks; ++cb) {
          uint8_t* cstage = smem_c + (blk_iter & 1u) * kCBlockBytes;
          uint32_t cbuf_u32 = ptx::smem_u32(cstage);
          if (p.use_tma_store) {       // the TMA store that last used this buffer must have finished reading it
            if (et == 0) ptx::bulk_wait_read<1>();
            __syncwarp();
            ptx::named_bar_sync(1, kEpiThreads);
          }
          // ---- TMEM -> registers -> 16-bit (or fp32 ring partial) -> swizzled smem ----
#pragma unroll
          for (int h = 0; h < kColsPerBlock / 32; ++h) {
            uint32_t v[32];
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) +
                                   static_cast<uint32_t>(acc * BN + cb * kCBlockCols + h * 32);
            ptx::tmem_ld_32x32b_x32(taddr, v);
            ptx::tmem_ld_wait();
            float f[32];
            if (p.in_kind == 1) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = static_cast<float>(static_cast<int>(v[i]));      // int32 accumulators
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
            }
            if (p.scale_a != nullptr || p.scale_b != nullptr) {       // dequantise: C = acc * scale_a[row] * scale_b[col]
              const int grow = row_base + my_row, gcol = col_base + cb * kCBlockCols + h * 32;
              const float sa = (kMode == kAG && p.ag_scale_ws != nullptr) ? ag_row_sa
                               : (p.scale_a != nullptr && grow < p.M) ? p.scale_a[grow] : 1.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] *= sa * ((p.scale_b != nullptr && gcol + i < p.N) ? p.scale_b[gcol + i] : 1.f);
            }
            if (p.row_scale != nullptr) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] *= row_scale;
            }
            if (sk_n > 0) {
              const int ch = cb * (kColsPerBlock / 32) + h;
              for (int pp = 0; pp < sk_n; ++pp) {
                const size_t pidx = static_cast<size_t>(un.slot * (p.sk_parts - 1) + pp) * kCtaGroup + cta_rank;
                const float* src = p.sk_ws + pidx * (BM * BN) + (ch * 4 + ew) * 1024 + lane * 4;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                  const uint4 x = ptx::ld_relaxed_sys_v4(src + q * 128);
                  f[4 * q] += __uint_as_float(x.x); f[4 * q + 1] += __uint_as_float(x.y);
                  f[4 * q + 2] += __uint_as_float(x.z); f[4 * q + 3] += __uint_as_float(x.w);
                }
              }
            }
            if constexpr (kMode == kRS) {
              if (rs_step > 0) {   // add the running partial pushed by rank+1 (same global coordinates)
                const int grow = row_base + my_row;
                const int gcol = col_base + cb * kCBlockCols + h * 32;
                if (grow < p.M && f32_in) {
                  const char* src = rs_in + (static_cast<size_t>(grow) * p.N + gcol) * 4;
#pragma unroll
                  for (int q = 0; q < 8; ++q) {
                    if (gcol + q * 4 < p.N) {
                      const uint4 x = ptx::ld_relaxed_sys_v4(src + q * 16);
                      f[4 * q] += __uint_as_float(x.x); f[4 * q + 1] += __uint_as_float(x.y);
                      f[4 * q + 2] += __uint_as_float(x.z); f[4 * q + 3] += __uint_as_float(x.w);
                    }
                  }
                } else if (grow < p.M) {
                  const char* src = rs_in + (static_cast<size_t>(grow) * p.N + gcol) * 2;
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    if (gcol + q * 8 < p.N) {
                      const uint4 x = ptx::ld_relaxed_sys_v4(src + q * 16);
                      const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                      for (int e = 0; e < 4; ++e) {
                        if (p.in_is_bf16) {
                          f[q * 8 + 2 * e] += ptx::bf16_lo(w[e]);
                          f[q * 8 + 2 * e + 1] += ptx::bf16_hi(w[e]);
                        } else {
                          const __half2 hh = *reinterpret_cast<const __half2*>(&w[e]);
                          f[q * 8 + 2 * e] += __low2float(hh);
                          f[q * 8 + 2 * e + 1] += __high2float(hh);
                        }
                      }
                    }
                  }
                }
              }
            }
            if (kMode == kRS && f32_out) {
              // fp32 ring partial: these 32 columns are one 128-byte row of their own staging block (own smem buffer)
              if (h > 0) { ++blk_iter; cbuf_u32 = ptx::smem_u32(smem_c + (blk_iter & 1u) * kCBlockBytes); }
#pragma unroll
              for (int q = 0; q < 8; ++q)
                ptx::st_shared_v4(cbuf_u32 + my_row * 128 + ((q ^ (my_row & 7)) << 4),
                                  make_uint4(__float_as_uint(f[4 * q]), __float_as_uint(f[4 * q + 1]), __float_as_uint(f[4 * q + 2]), __float_as_uint(f[4 * q + 3])));
              if (cb == kNumCBlocks - 1 && h == kColsPerBlock / 32 - 1) {
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                  if constexpr (kCtaGroup == 1) ptx::mbar_arrive(tmem_empty + acc);
                  else ptx::mbar_arrive_cluster(tmem_empty + acc, 0);
                }
              }
              ptx::named_bar_sync(1, kEpiThreads);
              const int gcol = col_base + cb * kCBlockCols + h * 32 + (et & 7) * 4;
#pragma unroll
              for (int r = et >> 3; r < BM; r += kEpiThreads / 8) {
                const int grow = row_base + r;
                if (grow < p.M && gcol < p.N) {
                  const uint4 o = ptx::ld_shared_v4(cbuf_u32 + r * 128 + (((et & 7) ^ (r & 7)) << 4));
                  ptx::st_v4(dst_base + (static_cast<size_t>(grow - dst_row_off) * dst_ld + gcol) * 4, o);
                }
              }
              continue;
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint4 o;
              if (p.in_is_bf16) {
                o.x = ptx::pack_bf16x2(f[q * 8 + 0], f[q * 8 + 1]); o.y = ptx::pack_bf16x2(f[q * 8 + 2], f[q * 8 + 3]);
                o.z = ptx::pack_bf16x2(f[q * 8 + 4], f[q * 8 + 5]); o.w = ptx::pack_bf16x2(f[q * 8 + 6], f[q * 8 + 7]);
              } else {
                o.x = ptx::pack_f16x2(f[q * 8 + 0], f[q * 8 + 1]); o.y = ptx::pack_f16x2(f[q * 8 + 2], f[q * 8 + 3]);
                o.z = ptx::pack_f16x2(f[q * 8 + 4], f[q * 8 + 5]); o.w = ptx::pack_f16x2(f[q * 8 + 6], f[q * 8 + 7]);
              }
              const int chunk = h * 4 + q;                                   // 16-byte chunk inside the 128-byte row
              ptx::st_shared_v4(cbuf_u32 + my_row * 128 + ((chunk ^ (my_row & 7)) << 4), o);
            }
          }
          ++blk_iter;
          if (kMode == kRS && f32_out) continue;     // fp32 partial already stored block by block
          if (cb == kNumCBlocks - 1) {
            // accumulator fully read: hand the TMEM stage back to the MMA issuer (on the leader CTA)
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (kCtaGroup == 1) ptx::mbar_arrive(tmem_empty + acc);
              else ptx::mbar_arrive_cluster(tmem_empty + acc, 0);
            }
          }
          if (p.use_tma_store) ptx::fence_proxy_async_smem();
          ptx::named_bar_sync(1, kEpiThreads);
          // ---- smem -> global ----
          const int gcol0 = col_base + cb * kCBlockCols;
          if (p.use_tma_store) {
            if (et == 0 && gcol0 < p.N && row_base < p.M) {
              ptx::tma_store_3d(&p.tmap_c, cstage, gcol0, row_base, cbuf_u);
              ptx::bulk_commit();
            }
            __syncwarp();
          } else {
            // 8 lanes cover one 128-byte row: fully coalesced 16-byte stores (NVLink-friendly for peer pointers)
            constexpr int kChunks = kColsPerBlock / 8;            // 16-byte chunks per row that carry data
            const int chunk = et & 7;
#pragma unroll
            for (int r = et >> 3; r < BM; r += kEpiThreads / 8) {
              const int grow = row_base + r;
              const int gcol = gcol0 + chunk * 8;
              if (chunk < kChunks && grow < p.M && gcol < p.N) {
                int drow = grow - dst_row_off;
                if (p.c_scatter) { drow = p.c_scatter[grow]; if (drow < 0 || drow == p.a_gather_pad) continue; }
                const uint4 o = ptx::ld_shared_v4(cbuf_u32 + r * 128 + ((chunk ^ (r & 7)) << 4));
                if constexpr (kMode == kEPC) {
                  const uint32_t v = p.c_route[grow];               // return address delivered by the dispatch
                  if (v == 0xffffffffu) continue;
                  char* rb = symm_at(p.symm, p.rs_stage + (ph & 1u) * p.rs_stage_buf_bytes, static_cast<int>(v >> 24));
                  ptx::st_v4(rb + (static_cast<size_t>(v & 0xffffffu) * p.N + gcol) * 2, o);
                } else if constexpr (kMode == kMoeRS) {
                  char* d = dst_base + (static_cast<size_t>(drow / p.mrs_topk) * dst_ld + gcol) * 2;     // pair id -> token row
                  if (p.in_is_bf16) ptx::red_add_bf16x8(d, o); else ptx::red_add_f16x8(d, o);
                } else {
                  ptx::st_v4(dst_base + (static_cast<size_t>(drow) * dst_ld + gcol) * 2, o);
                }
              }
            }
          }
        }
        if (sk_n > 0) {      // partials consumed: re-arm the flags for the next launch
          ptx::named_bar_sync(2, kEpiThreads);
          if (et < sk_n) p.sk_flags[static_cast<size_t>(un.slot * (p.sk_parts - 1) + et) * kCtaGroup + cta_rank] = 0u;
        }
        if constexpr (kMode == kRS) {
          if (!rs_final) {
            // all epilogue threads' stores for this tile are issued -> one thread publishes the tile to rank-1
            ptx::named_bar_sync(2, kEpiThreads);
            if (et == 0) {
              const int W = p.symm.world, me = p.symm.rank;
              uint32_t* f = p.rs_flags + (ph & 1u) * total_tiles + m_tile * p.num_n + n_tile;
              ptx::fence_acq_rel_sys();
              ptx::st_release_sys(symm_at(p.symm, f, (me - 1 + W) % W), ph);
            }
            __syncwarp();
          }
        }
        if constexpr (kMode == kMoeRS) {
          // this CTA tile has been added to the partial: count it for its column chunk; whoever completes the chunk tells every
          // rank (release at system scope, cumulative over all CTAs' reductions through the gpu-scope counter)
          ptx::named_bar_sync(2, kEpiThreads);
          if (et == 0) {
            int c = 0;
            while (c + 1 < p.mrs_n_chunks && n_tile >= p.mrs_chunk_start[c + 1]) ++c;
            const uint32_t expected = static_cast<uint32_t>(*p.mrs_total_padded / BM) * (p.mrs_chunk_start[c + 1] - p.mrs_chunk_start[c]);
            __threadfence();
            if (ptx::atom_add_acq_rel_gpu(p.mrs_counter + (ph & 1u) * (p.mrs_n_chunks + 1) + c, 1u) == expected - 1u) {
              const int W = p.symm.world, me = p.symm.rank;
              uint32_t* f = p.rs_flags + (static_cast<size_t>(ph & 1u) * p.mrs_n_chunks + c) * W + me;
              ptx::fence_acq_rel_sys();
              for (int d = 0; d < W; ++d) ptx::st_relaxed_sys(symm_at(p.symm, f, (me + d) % W), ph);
            }
          }
          __syncwarp();
        }
        if constexpr (kMode == kAR) {
          // each CTA of a pair stages its own 128 rows and publishes its own flag word (index carries the CTA rank);
          // the consumer waits for every (row half, source rank) word of the tile
          ptx::named_bar_sync(2, kEpiThreads);
          if (et == 0 && p.a2a_cols_per_rank > 0) {
            // count finished 128-row blocks per destination; the last one tells that rank "all of my rows have landed"
            const int W = p.symm.world, me = p.symm.rank;
            const uint32_t per_dst = static_cast<uint32_t>(p.num_m * kCtaGroup * (p.a2a_cols_per_rank / BN));
            ptx::fence_acq_rel_sys();
            if (ptx::atom_add_acq_rel_gpu(p.a2a_count + a2a_dst, 1u) == per_dst - 1u) {
              p.a2a_count[a2a_dst] = 0;
              ptx::fence_acq_rel_sys();
              ptx::st_release_sys(symm_at(p.symm, p.rs_flags + (ph & 1u) * W + me, a2a_dst), ph);
            }
          } else if (et == 0) {
            const int W = p.symm.world, me = p.symm.rank;
            uint32_t* f = p.rs_flags + static_cast<size_t>(ph & 1u) * p.rs_flag_tiles * W +
                          static_cast<size_t>((m_tile * kCtaGroup + static_cast<int>(cta_rank)) * p.num_n + n_tile) * W + me;
            ptx::fence_acq_rel_sys();
            for (int d = 0; d < W; ++d) ptx::st_relaxed_sys(symm_at(p.symm, f, (me + d) % W), ph);
          }
          __syncwarp();
        }
        if (lane == 0) prof_record(p.prof, static_cast<int>(blockIdx.x) * 8 + warp, 5, false);
        if (++acc == kAccStages) { acc = 0; acc_phase ^= 1u; }
      }
      if (p.use_tma_store && et == 0) ptx::bulk_wait<0>();
      __syncwarp();
      if constexpr (kMode == kEPC) {
        // my rows have been stored to their owners: make them visible system wide before this CTA counts itself out
        ptx::named_bar_sync(2, kEpiThreads);
        if (et == 0) ptx::fence_acq_rel_sys();
      }
    }

    // ---- teardown ----
    ptx::tc_fence_before();
    if constexpr (kCtaGroup == 2) ptx::cluster_sync(); else __syncthreads();
    if (warp == 2) ptx::tmem_dealloc<kCtaGroup>(tmem_base, kTmemCols);
  }

  // ---- phase bookkeeping: the last CTA to leave advances the call counter ----
  if constexpr (kMode != kPlain) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(p.phase + 1, 1u) == gridDim.x - 1) {
        p.phase[1] = 0;
        __threadfence();
        p.phase[0] = ph;
        if constexpr (kMode == kEPC) {     // every CTA fenced its stores (sys scope) before counting out: tell all owners
          ptx::fence_acq_rel_sys();
          for (int d = 0; d < p.symm.world; ++d)
            ptx::st_release_sys(symm_at(p.symm, p.rs_flags + (ph & 1u) * p.symm.world + p.symm.rank, d), ph);
        }
      }
    }
  }
}

}  // namespace gemm
}  // namespace td
