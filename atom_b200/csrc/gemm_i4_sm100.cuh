// gemm_i4_sm100.cuh -- W4A4 group-quantised GEMM with INT8 keeper for B200 (sm_100a).
//
// Replaces the reference's compute_gemm_imma / DenseLayerGEMM_i4[_o4]_kernel
// (/root/reference/kernels/include/GEMM/Dense_layer_gemm_i4_o16.cuh:436-710,
//  /root/reference/e2e/punica-atom/punica/ops/csrc/GEMM/DenseLayerGEMM_i4_o4.cu:440-787).
// Same operands, same layouts, same arithmetic (exact INT32 group sums, one FP16 multiply of the
// two scales, FP32 fma accumulation in group order, keeper last, RN cast to half) -- different machine:
//
//   TMA (packed INT4 tiles, 64 B rows)  ->  smem "packed ring"
//   converter warps: nibble -> INT8 (value*16, no sign-extension work) into the canonical
//       K-major SWIZZLE_128B operand layout ("expanded ring"); the INT8 keeper group is TMA'd straight
//       into that layout.  Blackwell has no INT4 MMA: kind::i8 is the integer tensor path.
//   one thread: tcgen05.mma.kind::i8  (128 x BN x 32) x 4 per 128-wide quantisation group, INT32 in TMEM
//   epilogue warpgroups: tcgen05.ld -> acc += float(c) * half(sA*sB) in registers, overlapped with the
//       MMAs of the following stage; FP16 (o16) or asymmetric INT4 (o4) output.
//
// A pipeline STAGE is GS quantisation groups, not one: measured on B200 (tools/sync_bench.cu) a warp-to-warp mbarrier
// hand-off costs ~180 cycles one way, a wait on an already completed phase ~100, a tcgen05.commit ~200 of the issuing
// thread -- against 256 tensor cycles for one 128x128x128 group.  Every hand-off (TMA->converter->MMA->epilogue) and
// every commit therefore covers GS groups; one commit per stage serves both the epilogue ("accumulators ready") and
// the converter ("operand slot free").
//
// Weight-stationary: MMA-M = 128 output channels (B), MMA-N = BN = 64 tokens (A), 8 converter warps, 2 epilogue
// warpgroups.  gemm_dispatch runs it for 33-128 tokens; optionally split along K over a thread-block cluster, partial
// sums pushed into the leader through DSMEM.
//
// GemmArgs, expand_chunk, convert_tile, the scale layout and trace_stamp are shared with the decode and 128x128 kernels.
#pragma once
#include "ptx_sm100.cuh"

namespace atom {

struct GemmArgs {
  const __half* a_scale;         // [G][S(M)]  ldmatrix-replicated layout (Reorder.cuh:39-50)
  const __half* b_scale;         // [G][N]
  const __half* a_keeper_scale;  // [S(M)]
  const __half* b_keeper_scale;  // [N]
  __half* d;                     // o16: [M][N]
  uint8_t* d4;                   // o4 : [M][N/2]
  __half2* d_scale;              // o4 : [M][N/128] (scale, zero)
  uint8_t* d4_v;                 // fused q/k/v projection (decode kernel, EPI_QKV): channel tiles [0, seg_tiles) are q -> d (o16),
  __half2* d_scale_v;            //   [seg_tiles, 2 seg_tiles) are k -> d4 / d_scale (o4), the rest v -> d4_v / d_scale_v (o4)
  int seg_tiles;
  // fused gate/up projection + SiLU(gate)*up + dynamic quantisation (decode kernel, EPI_GATEUP): the activation 4-tuple
  // that activate_fp16_i4 would have produced (Activate.cuh:67-180); gu_rows = intermediate size I (up rows start at I)
  int8_t* q8_out; uint8_t* q4_out; __half* q8_scale; __half* q4_scale; int gu_rows;
  int ldb_scale;                 // pitch (halves) of the b_scale rows; N unless the weights are a slice of a fused matrix
  int M, N, G;                   // G = number of INT4 groups = K/128 - 1
  int lda_scale;                 // S(M)
  unsigned long long* trace;     // optional device buffer [ctas][128] of clock64 stamps (atom_gemm_set_trace), else null
  const uint8_t* a4;             // packed INT4 activations [M][(K-128)/2] and their INT8 keeper [M][128]: the decode kernel
  const int8_t* a8;              //   reads the (tiny) token operand straight from global memory instead of through TMA
  int pdl;                       // launched with programmatic stream serialization: weights may be fetched before the
                                 // preceding kernel has finished, everything that reads activations waits (griddepcontrol)
  int dbg;                       // ATOM_B200_GU_MODE experiment bits (gate/up hand-off), 0 in production
  ArArgs ar;                     // row-parallel projection (tp.py): ar.bufs != null => the decode kernel's o16 epilogue stores D
                                 // into slot [call % 3][rank] of every rank's receive buffer instead of d (push half of the
                                 // all-reduce, comm_kernels.cuh); the consumer is rmsnorm_quant_kernel's reducing variant
};

// timeline stamps for pipeline debugging (tools/gpu_check.py trace): slot layout per CTA
//   0 start | 1 setup done | 2 epilogue loop done | 3 reduction done | 4 end
//   per stage s < 16 (8 for the last row): 8+s producer issued | 24+s converter got its operand slot |
//   40+s converter saw the packed tiles | 56+s conversion stored | 72+s converter fenced+arrived | 88+s MMA thread woke |
//   104+s accumulators ready (epilogue) | 120+s epilogue done
__device__ __forceinline__ void trace_stamp(const GemmArgs& a, int slot) {
  if (a.trace != nullptr && slot < 128) {
    const int cta = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    a.trace[(size_t)cta * 128 + slot] = (unsigned long long)clock64();
  }
}

__device__ __forceinline__ float silu_ref(float x) { return x / (1.0f + expf(-x)); }   // Activate.cuh:28
__host__ __device__ __forceinline__ int scale_index(int row) { return (row / 16) * 64 + (row % 8) * 8 + ((row / 8) % 2); }
__host__ __device__ __forceinline__ int scale_size(int m) { return m / 16 * 64 + 64 - (1 - (m % 16) / 8) * (8 - (m % 8)) * 8; }

template <int GS, int kPack, int kSplit, bool kO4>
struct GemmCfg {
  static constexpr int BM = 128;                                  // MMA M (TMEM lanes) = output channels per tile
  static constexpr int BN = 64;                                   // MMA N = tokens per tile
  static constexpr int RING = 2;                                  // operand-slot / accumulator stages
  static constexpr int TMEM_COLS_RAW = RING * GS * BN;
  static constexpr int TMEM_COLS = TMEM_COLS_RAW <= 32 ? 32 : (TMEM_COLS_RAW <= 64 ? 64 : (TMEM_COLS_RAW <= 128 ? 128 : (TMEM_COLS_RAW <= 256 ? 256 : 512)));
  static constexpr int SCALE_STAGES = 4;                          // scale ring depth, in stages
  static constexpr int SCALE_GROUP_BYTES = 512;                   // 256 B MMA-M side + 256 B MMA-N side, raw copies
  static constexpr int EPI_WGS = 2;                               // epilogue warpgroups (each owns BN/EPI_WGS columns)
  static constexpr int CPT = BN / EPI_WGS;                        // accumulator columns per epilogue thread
  static constexpr int CONV_WARPS = 8;
  static constexpr int CONV_THREADS = CONV_WARPS * 32;
  static constexpr int THREADS = 256 + 128 * EPI_WGS + (CONV_WARPS - 4) * 32;   // extra converters sit after the epilogue
  static constexpr int PACK_P = BM * 64, PACK_Q = BN * 64;        // bytes per packed group
  static constexpr int EXP_P = BM * 128, EXP_Q = (BN * 128 + 1023) / 1024 * 1024;   // bytes per expanded group
  static constexpr int OFF_EXP_P = 0;
  static constexpr int OFF_EXP_Q = OFF_EXP_P + RING * GS * EXP_P;
  static constexpr int OFF_PACK_P = OFF_EXP_Q + RING * GS * EXP_Q;
  static constexpr int OFF_PACK_Q = OFF_PACK_P + kPack * GS * PACK_P;
  static constexpr int OFF_SM = OFF_PACK_Q + kPack * GS * PACK_Q; // scale ring (16-B aligned)
  static constexpr int RED_BYTES = BM * BN * 4;                   // one rank's split-K partial [col][row] fp32
  static constexpr int OFF_RED = OFF_SM + SCALE_STAGES * GS * SCALE_GROUP_BYTES;   // leader only: pushed partials
  static constexpr int OFF_BAR = OFF_RED + (kSplit > 1 ? (kSplit - 1) * RED_BYTES : 0);
  static constexpr int NUM_BARS = 2 * kPack + 3 * RING + 2 * SCALE_STAGES;
  static constexpr int OFF_TMEM_PTR = OFF_BAR + NUM_BARS * 8;
  static constexpr int SMEM_BYTES = OFF_TMEM_PTR + 16 + 1024;     // + slack for the 1024-B alignment fix-up
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static_assert(TMEM_COLS_RAW <= 512, "TMEM has 512 columns");
};

// nibble -> int8(value * 16): element 2b of the word lands in byte b of `lo`, element 2b+1 in byte b of `hi`.
// The same permutation of K inside a 32-element chunk is applied to both operands, so dot products are unchanged;
// the uniform factor 16*16 = 256 is carried by the accumulator and removed exactly at the output cast.
__device__ __forceinline__ void expand_chunk(const uint4& w, uint4& lo, uint4& hi) {
  lo.x = (w.x << 4) & 0xF0F0F0F0u; hi.x = w.x & 0xF0F0F0F0u;
  lo.y = (w.y << 4) & 0xF0F0F0F0u; hi.y = w.y & 0xF0F0F0F0u;
  lo.z = (w.z << 4) & 0xF0F0F0F0u; hi.z = w.z & 0xF0F0F0F0u;
  lo.w = (w.w << 4) & 0xF0F0F0F0u; hi.w = w.w & 0xF0F0F0F0u;
}

// convert `rows` packed rows (64 B each, dense) into the K-major SWIZZLE_128B layout (128 B rows, 8-row atoms).
// All of a thread's 16-B chunks are loaded before any is expanded/stored so that the LDS latencies overlap.
template <int kRows, int kThreads>
__device__ __forceinline__ void convert_tile(const uint8_t* __restrict__ packed, uint8_t* __restrict__ expanded, int t) {
  constexpr int kChunks = kRows * 4;
  constexpr int kIter = (kChunks + kThreads - 1) / kThreads;
  uint4 w[kIter];
#pragma unroll
  for (int i = 0; i < kIter; ++i) {
    const int c = t + i * kThreads;
    if (kChunks % kThreads == 0 || c < kChunks) w[i] = *reinterpret_cast<const uint4*>(packed + c * 16);
  }
#pragma unroll
  for (int i = 0; i < kIter; ++i) {
    const int c = t + i * kThreads;
    if (kChunks % kThreads == 0 || c < kChunks) {
      const int r = c >> 2, j = c & 3;
      uint4 lo, hi;
      expand_chunk(w[i], lo, hi);
      uint8_t* row = expanded + (r >> 3) * 1024 + (r & 7) * 128;
      *reinterpret_cast<uint4*>(row + (((2 * j) ^ (r & 7)) << 4)) = lo;
      *reinterpret_cast<uint4*>(row + (((2 * j + 1) ^ (r & 7)) << 4)) = hi;
    }
  }
}

template <int GS, int kPack, int kSplit, bool kO4>
__global__ void __launch_bounds__(GemmCfg<GS, kPack, kSplit, kO4>::THREADS, 1)
gemm_i4_kernel(const __grid_constant__ CUtensorMap tm_p4,   // packed INT4 weights      (box 64 B x 128 rows)
               const __grid_constant__ CUtensorMap tm_q4,   // packed INT4 tokens       (box 64 B x BN rows)
               const __grid_constant__ CUtensorMap tm_p8,   // INT8 keeper, weights     (box 128 B x 128 rows, SW128)
               const __grid_constant__ CUtensorMap tm_q8,   // INT8 keeper, tokens      (box 128 B x BN rows, SW128)
               const GemmArgs args) {
  using C = GemmCfg<GS, kPack, kSplit, kO4>;
  constexpr int BN = C::BN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-B alignment (SWIZZLE_128B atoms) by offsetting the shared array, NOT by integer-casting the pointer:
  // an integer round trip makes the compiler fall back to generic LD/ST for every smem access.
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
  uint64_t* pack_full = bars;                          // TMA landed the stage's packed tiles          (1 + tx)
  uint64_t* pack_empty = pack_full + kPack;            // converters have read them                    (CONV_WARPS)
  uint64_t* exp_full = pack_empty + kPack;             // expanded operands of the stage are in place  (CONV_WARPS [+ tx])
  uint64_t* mma_done = exp_full + C::RING;             // the stage's MMAs completed: accumulators ready AND slot reusable (1)
  uint64_t* tmem_empty = mma_done + C::RING;           // epilogue has read the stage's accumulators   (4 * EPI_WGS)
  uint64_t* scale_full = tmem_empty + C::RING;         // scales of the stage landed                   (32, cp.async noinc)
  uint64_t* scale_empty = scale_full + C::SCALE_STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + C::OFF_TMEM_PTR);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // blockIdx.x = output-channel tile: CTAs launched together share the token tile (L2) and stream disjoint weights
  const int tile_ch = blockIdx.x, tile_tok = blockIdx.y;
  const int p0 = tile_ch * C::BM;                        // first row of the MMA-M operand (weights)
  const int q0 = tile_tok * BN;                          // first row of the MMA-N operand (tokens)
  const int m0 = q0, n0 = p0;                            // token / channel origin of the tile

  // K split over the cluster: groups [g_begin, g_end) of the G+1 groups (index G = INT8 keeper)
  const int total_groups = args.G + 1;
  int g_begin = 0, g_end = total_groups;
  uint32_t krank = 0;
  if constexpr (kSplit > 1) {
    krank = cluster_ctarank();
    const int per = (total_groups + kSplit - 1) / kSplit;
    g_begin = min((int)krank * per, total_groups);
    g_end = min(g_begin + per, total_groups);
  }
  const int iters = g_end - g_begin;                        // groups of this CTA
  const int nstages = (iters + GS - 1) / GS;
  // stage s covers groups g_begin + s*GS .. ; INT4 groups of a stage travel through the packed ring, the keeper
  // (only ever the last group of the last stage) goes straight to its operand slot
  auto stage_groups = [&](int s) { return min(GS, iters - s * GS); };
  auto stage_int4 = [&](int s) { const int g0 = g_begin + s * GS; return max(0, min(g0 + stage_groups(s), args.G) - g0); };
  if (threadIdx.x == 0) trace_stamp(args, 0);

  // ---------------------------------------------------------------- one-time setup
  // Thread 0 initialises the barriers and immediately fires the first kPack stages of TMA loads: the DRAM round trip
  // of the first tiles (the longest latency on the critical path of a decode-sized problem) then overlaps the TMEM
  // allocation and the CTA-wide sync instead of following them.
  // part: 0 = both operands; 1 = arm the barrier and load the WEIGHT tiles only; 2 = load the ACTIVATION tiles only
  // (PDL: the weights do not depend on the preceding kernel and are fetched before griddepcontrol.wait)
  auto issue_stage = [&](int s, int ps, int part = 0) {
    const int n4 = stage_int4(s);
    if (part != 2) mbar_arrive_expect_tx(&pack_full[ps], n4 * (C::PACK_P + C::PACK_Q));
    const bool do_p = part != 2, do_q = part != 1;      // P = weights, Q = activations
    for (int j = 0; j < n4; ++j) {
      const int g = g_begin + s * GS + j;
      if (do_p) tma_load_2d(smem + C::OFF_PACK_P + (ps * GS + j) * C::PACK_P, &tm_p4, &pack_full[ps], g * 64, p0);
      if (do_q) tma_load_2d(smem + C::OFF_PACK_Q + (ps * GS + j) * C::PACK_Q, &tm_q4, &pack_full[ps], g * 64, q0);
    }
    if (s < 16 && part != 1) trace_stamp(args, 8 + s);
  };
  int s_issued = 0;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_p4); tma_prefetch_desc(&tm_q4);
    // the barriers the first loads need come first; everything else is initialised while those loads are in flight
    for (int i = 0; i < kPack; ++i) mbar_init(&pack_full[i], 1);
    fence_barrier_init();
    if (!args.pdl) {
      for (; s_issued < kPack && s_issued < nstages && stage_int4(s_issued) > 0; ++s_issued) issue_stage(s_issued, s_issued);
    } else {
      griddep_launch_dependents();
      int s_w = 0;
      for (; s_w < kPack && s_w < nstages && stage_int4(s_w) > 0; ++s_w) issue_stage(s_w, s_w, 1);
      griddep_wait();                       // from here on the preceding kernel's output (the activations) may be read
      for (; s_issued < s_w; ++s_issued) issue_stage(s_issued, s_issued, 2);
    }
    tma_prefetch_desc(&tm_p8); tma_prefetch_desc(&tm_q8);
    for (int i = 0; i < kPack; ++i) mbar_init(&pack_empty[i], C::CONV_WARPS);
    for (int i = 0; i < C::RING; ++i) {
      mbar_init(&exp_full[i], C::CONV_WARPS); mbar_init(&mma_done[i], 1); mbar_init(&tmem_empty[i], 4 * C::EPI_WGS);
    }
    for (int i = 0; i < C::SCALE_STAGES; ++i) { mbar_init(&scale_full[i], 32); mbar_init(&scale_empty[i], 4 * C::EPI_WGS); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<C::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // split-K: a CTA's shared memory may only be written remotely once that CTA has started -- every thread arrives
  // here (cheap, non-blocking) and the epilogue warps wait right before their first st.shared::cluster
  if constexpr (kSplit > 1) cluster_arrive_relaxed();
  const uint32_t tmem_base = *tmem_ptr;
  if (threadIdx.x == 0) trace_stamp(args, 1);

  if (warp == 0) {
    // ============================================================ TMA producer (INT4 groups only)
    if (lane == 0) {
      for (int s = s_issued; s < nstages; ++s) {
        if (stage_int4(s) == 0) break;       // a trailing keeper-only stage has nothing in the packed ring
        const int ps = s % kPack;
        mbar_wait(&pack_empty[ps], ((s / kPack) & 1) ^ 1);
        issue_stage(s, ps);
      }
    }
  } else if (warp == 1) {
    // ============================================================ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_i8(C::BM, BN);
      for (int s = 0; s < nstages; ++s) {
        const int es = s % C::RING;
        if (s >= C::RING) mbar_wait(&tmem_empty[es], ((s / C::RING) - 1) & 1);
        mbar_wait(&exp_full[es], (s / C::RING) & 1);
        tc_fence_after();
        if (s < 16) trace_stamp(args, 88 + s);
        const int ng = stage_groups(s);
        for (int j = 0; j < ng; ++j) {
          const uint64_t dp = umma_desc_k_sw128(smem_u32(smem + C::OFF_EXP_P + (es * GS + j) * C::EXP_P));
          const uint64_t dq = umma_desc_k_sw128(smem_u32(smem + C::OFF_EXP_Q + (es * GS + j) * C::EXP_Q));
#pragma unroll
          for (int k = 0; k < 4; ++k)   // 4 x K=32 per 128-wide group; +32 B inside the swizzle atom per step
            umma_i8(tmem_base + (es * GS + j) * BN, dp + (uint64_t)(k * 2), dq + (uint64_t)(k * 2), idesc, k > 0);
        }
        umma_commit(&mma_done[es]);     // one commit per stage: epilogue may read, converter may refill
      }
    }
  } else if (warp == 3) {
    // ============================================================ scale loader: cp.async straight into the scale ring,
    // completion counted on scale_full by the copy engine -- no thread ever waits on a scale's DRAM latency.
    // Group slot layout (raw copies of the reference layouts):
    //   [0,256)   MMA-M side: 128 B-scale halves of the channel tile (thread n reads the pair word n/2)
    //   [256,512) MMA-N side: BN/16*8 (lower,upper) A-scale words of the token rows
    if (args.pdl) griddep_wait();           // the activation scales are the preceding kernel's output
    for (int s = 0; s < nstages; ++s) {
      const int ss = s % C::SCALE_STAGES;
      if (s >= C::SCALE_STAGES) mbar_wait(&scale_empty[ss], ((s / C::SCALE_STAGES) - 1) & 1);
      const int ng = stage_groups(s);
      for (int j = 0; j < ng; ++j) {
        const int g = g_begin + s * GS + j;
        const bool keeper = (g == args.G);
        const __half* as_row = keeper ? args.a_keeper_scale : args.a_scale + (size_t)g * args.lda_scale;
        const __half* bs_row = keeper ? args.b_keeper_scale : args.b_scale + (size_t)g * args.N;
        uint8_t* slot_p = smem + C::OFF_SM + (ss * GS + j) * C::SCALE_GROUP_BYTES;
        constexpr int TOK = BN, CHN = C::BM;
        uint8_t* tok_dst = slot_p + 256;
        uint8_t* chn_dst = slot_p;
#pragma unroll
        for (int w = lane; w < TOK / 2; w += 32) {              // A-scale words: rows (16 blk + i, 16 blk + i + 8)
          const int blk = w >> 3, i = w & 7;
          if (m0 + 16 * blk + i < args.M) cp_async_4(tok_dst + w * 4, as_row + 64 * (m0 / 16 + blk) + 8 * i);
        }
#pragma unroll
        for (int c = lane; c < CHN / 8; c += 32)                // B-scale: 8 channels per 16-B chunk
          if (n0 + 8 * c < args.N) cp_async_16(chn_dst + c * 16, bs_row + n0 + 8 * c);
      }
      cp_async_mbar_arrive_noinc(&scale_full[ss]);
    }
  } else if ((warp >= 4 && warp < 8) || warp >= 8 + 4 * C::EPI_WGS) {
    // ============================================================ converter warps
    const int t = (warp < 8 ? warp - 4 : warp - 8 - 4 * C::EPI_WGS + 4) * 32 + lane;
    if (args.pdl && t == 0) griddep_wait();   // thread 0 TMA-loads the activation keeper: the preceding kernel's output
    for (int s = 0; s < nstages; ++s) {
      const int es = s % C::RING, ps = s % kPack;
      const int ng = stage_groups(s), n4 = stage_int4(s);
      if (s >= C::RING) mbar_wait(&mma_done[es], ((s / C::RING) - 1) & 1);   // MMAs that read this slot have completed
      if (t == 0 && s < 16) trace_stamp(args, 24 + s);
      if (n4 > 0) {
        mbar_wait(&pack_full[ps], (s / kPack) & 1);
        if (t == 0 && s < 16) trace_stamp(args, 40 + s);
#pragma unroll
        for (int j = 0; j < GS; ++j) {
          if (j < n4) {
            convert_tile<C::BM, C::CONV_THREADS>(smem + C::OFF_PACK_P + (ps * GS + j) * C::PACK_P,
                                                 smem + C::OFF_EXP_P + (es * GS + j) * C::EXP_P, t);
            convert_tile<BN, C::CONV_THREADS>(smem + C::OFF_PACK_Q + (ps * GS + j) * C::PACK_Q,
                                              smem + C::OFF_EXP_Q + (es * GS + j) * C::EXP_Q, t);
          }
        }
        if (t == 0 && s < 16) trace_stamp(args, 56 + s);
        fence_proxy_async_smem();     // generic-proxy stores -> visible to tcgen05.mma operand fetch
      }
      __syncwarp();
      if (lane == 0) {
        if (n4 > 0) mbar_arrive(&pack_empty[ps]);
        if (n4 < ng && t == 0) {        // the keeper is this stage's last group: TMA it into its operand slot
          mbar_arrive_expect_tx(&exp_full[es], C::EXP_P + BN * 128);
          tma_load_2d(smem + C::OFF_EXP_P + (es * GS + n4) * C::EXP_P, &tm_p8, &exp_full[es], 0, p0);
          tma_load_2d(smem + C::OFF_EXP_Q + (es * GS + n4) * C::EXP_Q, &tm_q8, &exp_full[es], 0, q0);
        } else {
          mbar_arrive(&exp_full[es]);
        }
      }
      if (t == 0 && s < 16) trace_stamp(args, 72 + s);
    }
  } else if (warp >= 8 && warp < 8 + 4 * C::EPI_WGS) {
    // ============================================================ epilogue warpgroup(s)
    const int wq = warp & 3;                       // TMEM lane quarter this warp may access
    const int row = wq * 32 + lane;                // MMA-M row == TMEM lane
    const int colbase = ((warp - 8) >> 2) * C::CPT;
    float acc[C::CPT];
#pragma unroll
    for (int i = 0; i < C::CPT; ++i) acc[i] = 0.f;

    for (int s = 0; s < nstages; ++s) {
      const int es = s % C::RING, ss = s % C::SCALE_STAGES;
      const int ng = stage_groups(s);
      mbar_wait(&scale_full[ss], (s / C::SCALE_STAGES) & 1);
      mbar_wait(&mma_done[es], (s / C::RING) & 1);
      tc_fence_after();
      if (warp == 8 && lane == 0 && s < 16) trace_stamp(args, 104 + s);
      for (int j = 0; j < ng; ++j) {
        const bool keeper = (g_begin + s * GS + j == args.G);
        const uint8_t* slot_p = smem + C::OFF_SM + (ss * GS + j) * C::SCALE_GROUP_BYTES;
        const __half2 sm2 = reinterpret_cast<const __half2*>(slot_p)[row >> 1];     // {sB[n&~1], sB[n|1]}
        // (lower, upper) A-scale words of this thread's token columns
        const __half2* snw = reinterpret_cast<const __half2*>(slot_p + 256) + (colbase >> 4) * 8;
        const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)((es * GS + j) * BN + colbase);
        constexpr int CH = (C::CPT >= 32) ? 32 : 16;
#pragma unroll
        for (int c0 = 0; c0 < C::CPT; c0 += CH) {
          uint32_t r[CH];
          if constexpr (CH == 32) tmem_ld_32x32b_x32(taddr + c0, r); else tmem_ld_32x32b_x16(taddr + c0, r);
          tmem_ld_wait();
          if (c0 + CH == C::CPT && j == ng - 1) {   // the stage's accumulators are in registers: hand TMEM back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[es]);
          }
          // INT4 groups carry a factor 256 (both operands are value*16); lift the keeper to the same domain
          if (keeper) {
#pragma unroll
            for (int i = 0; i < CH; ++i) r[i] = (uint32_t)((int32_t)r[i] << 8);
          }
          // thread = channel row (sm2 = {sB[n&~1], sB[n|1]}); columns = tokens, 16-aligned tile origin:
          // token i with i%16<8 pairs with sm2.x, i%16>=8 with sm2.y
#pragma unroll
          for (int q = 0; q < CH; q += 16) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const __half2 a2 = snw[((c0 + q) >> 4) * 8 + i];      // (sA[token q+i], sA[token q+i+8])
              const float2 rs = __half22float2(__hmul2(a2, sm2));
              acc[c0 + q + i] = fmaf((float)(int32_t)r[q + i], rs.x, acc[c0 + q + i]);
              acc[c0 + q + i + 8] = fmaf((float)(int32_t)r[q + i + 8], rs.y, acc[c0 + q + i + 8]);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&scale_empty[ss]);       // this warp no longer reads the stage's scales
      if (warp == 8 && lane == 0 && s < 8) trace_stamp(args, 120 + s);
    }
    if (warp == 8 && lane == 0) trace_stamp(args, 2);

    // ------------------------------------------------------------ split-K: push partials into the leader's smem
    // Remote stores need no round trip (a pull would put several DSMEM read latencies on the critical path); one
    // cluster barrier (release / acquire) publishes them, then only the leader goes on.
    if constexpr (kSplit > 1) {
      cluster_wait();                 // pairs with the setup arrive: every CTA of the cluster is running
      if (krank != 0) {
        const uint32_t remote = mapa_shared(smem_u32(smem + C::OFF_RED), 0) + (krank - 1) * C::RED_BYTES;
#pragma unroll
        for (int i = 0; i < C::CPT; ++i) st_dsmem_f32(remote + ((colbase + i) * C::BM + row) * 4, acc[i]);
      }
      cluster_arrive(); cluster_wait();
      if (krank == 0) {
        const float* red = reinterpret_cast<const float*>(smem + C::OFF_RED);
#pragma unroll
        for (int rk = 0; rk < kSplit - 1; ++rk) {
#pragma unroll
          for (int i = 0; i < C::CPT; ++i) acc[i] += red[rk * (C::RED_BYTES / 4) + (colbase + i) * C::BM + row];
        }
      }
    }
    if (warp == 8 && lane == 0) trace_stamp(args, 3);
    // ------------------------------------------------------------ output
    if (kSplit == 1 || krank == 0) {
      constexpr float kInv = 1.0f / 256.0f;   // exact: removes the 16*16 operand factor
      if constexpr (!kO4) {
        const int n = n0 + row;
        if (n < args.N) {
#pragma unroll
          for (int i = 0; i < C::CPT; ++i) {
            const int m = m0 + colbase + i;
            if (m < args.M) args.d[(size_t)m * args.N + n] = __float2half_rn(acc[i] * kInv);   // warp writes 64 B runs
          }
        }
      } else {
        // o4 epilogue (DenseLayerGEMM_i4_o4.cu:705-787): per (token, 128-channel head) asymmetric INT4 with the
        // reference's |v| min/max.  Thread = channel; reduce |v| min/max over the 128 channels of the head for every
        // token column.
        float* xch = reinterpret_cast<float*>(smem + C::OFF_PACK_P);   // packed ring is idle by now
        float* xmx = xch;                 // [4 warps][BN]
        float* xmn = xch + 4 * BN;
        const int ewarp = warp - 8;       // each of the 2 WGs owns CPT token columns
#pragma unroll
        for (int i = 0; i < C::CPT; ++i) {
          acc[i] *= kInv;
          // |v| >= 0: IEEE bit patterns order like unsigned integers, so one REDUX each replaces 5 shuffle rounds
          uint32_t ua = __float_as_uint(fabsf(acc[i])), umx = ua, umn = ua;
          if (n0 + row >= args.N) { umx = 0u; umn = 0x7f800000u; }
          umx = __reduce_max_sync(0xffffffffu, umx);
          umn = __reduce_min_sync(0xffffffffu, umn);
          if (lane == 0) { xmx[(ewarp & 3) * BN + colbase + i] = __uint_as_float(umx); xmn[(ewarp & 3) * BN + colbase + i] = __uint_as_float(umn); }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(128 * C::EPI_WGS) : "memory");
        const int n = n0 + row;
#pragma unroll
        for (int i = 0; i < C::CPT; ++i) {
          const int c = colbase + i, m = m0 + c;
          const float mx = fmaxf(fmaxf(xmx[c], xmx[BN + c]), fmaxf(xmx[2 * BN + c], xmx[3 * BN + c]));
          const float mn = fminf(fminf(xmn[c], xmn[BN + c]), fminf(xmn[2 * BN + c], xmn[3 * BN + c]));
          const float scale = (mx - mn) / 15.f, zero = -mn, r_scale = 1.f / scale;
          int q = (int)roundf((acc[i] + zero) * r_scale) & 0xF;
          const int qn = __shfl_down_sync(0xffffffffu, q, 1);     // channel n+1 lives in the next lane
          if (m < args.M && n < args.N) {
            if ((lane & 1) == 0) args.d4[(size_t)m * (args.N / 2) + n / 2] = (uint8_t)(q | (qn << 4));
            if (row == 0) args.d_scale[(size_t)m * (args.N / 128) + tile_ch] = __floats2half2_rn(scale, zero);
          }
        }
      }
    }
  }

  // ---------------------------------------------------------------- teardown
  if constexpr (kSplit > 1) {
    if (!(warp >= 8 && warp < 8 + 4 * C::EPI_WGS)) { cluster_wait(); cluster_arrive(); cluster_wait(); }   // setup phase, then the epilogue's publish phase
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<C::TMEM_COLS>(tmem_base);
  if (threadIdx.x == 0) trace_stamp(args, 4);
}

}  // namespace atom
