// Fused front of the shared-MLP chain (bf16 tier): one persistent kernel computes, per 256-point tile
// of a CTA pair,
//     conv1 (fp32 FMA) -> conv2 -> conv3 -> conv4        (src/model.py:43-46, BatchNorm folded, ReLU)
//     gate layer 1 (fp32 FMA)                            (src/model.py:33-34)
// with every intermediate activation kept in shared memory in the 128-byte-swizzled K-major layout that
// both UMMA (as the next layer's A operand) and TMA (as the source of the store into the operand row)
// understand.  Only the folded weights stream through TMA; every output (feat1..feat4, gate hidden block)
// leaves through TMA stores of [128 x 64] blocks (feat4 is staged in blocks that are idle at that point:
// 16-byte pieces of 32 different rows per store instruction cost 19k cycles per tile).  Compared with one GEMM
// launch per layer this removes the HBM round trip of feat1..feat3 as inputs and four launches per wave.
//
//   warp 0      : TMA producer for the weight k-blocks (both CTAs; bytes counted on the leader's barrier)
//   warp 1      : TMEM allocator (both CTAs) + tcgen05.mma.cta_group::2 issuer (leader)
//   warps 2..9  : compute warps: conv1 / gate layer 1 in fp32, and every layer's epilogue
//                 (TMEM -> bias + ReLU -> bf16 -> swizzled smem block).  Warp w owns TMEM lane quarter
//                 (w & 3) and column half ((w - 2) >> 2).
//
// TMEM: two 256-column accumulator buffers.  conv2 -> buf0[0:128), conv3 -> buf1, conv4 chunk 0 -> buf0,
// conv4 chunk 1 -> buf1, so conv4's second chunk runs while the first one is drained.  The next tile's conv1 and
// gate layer 1 are computed by the epilogue warps in the shadow of conv5 (between its chunk drains).
//
// conv5 (512 -> 1024, src/model.py:47; 75 % of the chain's FLOPs) runs in the same kernel with its A operand in
// TENSOR MEMORY: the conv4 epilogue writes feat4 as packed bf16 into TMEM columns [0, 256) (row = lane,
// two channels per column) besides staging it for the TMA store, and conv5 runs as
// tcgen05.mma.cta_group::2 [D], [A_tmem], B_desc ("TS" form) over eight 128-channel chunks that alternate between
// two accumulators (columns [256, 384) / [384, 512)): the drain of chunk n hides under the MMAs of chunk n + 1.
// An N = 128 TS MMA takes 77 cycles against 64 of math (tools/mma_probe.cu), but four 256-channel chunks through
// the single accumulator that fits beside feat4 serialise MMAs and drains (8.6k instead of 2 x 2.5k cycles per 256
// channels).  Only the weights touch shared memory: conv5 streams 512 KB of them per CTA and tile, and while it runs
// the four F2 / Z blocks (idle then) serve as four more 16 KB weight stages (7 in flight; one stage = two 64-wide
// k-blocks of the CTA's 64 weight rows = 8 MMAs per barrier round trip).  The F1 / GH blocks, idle from the end of conv2
// until the next tile's conv1, take the tile's first two conv5 stages ~10k cycles ahead of time, so conv5 starts with
// weights in place (a TMA round trip under load is ~2.8k cycles).  conv4 has the same problem at a smaller scale - eight
// k-blocks consumed in ~0.5k cycles each through three dedicated stages - so two of its first chunk's k-blocks land in
// the Z blocks (idle until that chunk's drain stages feat4 through them): five k-blocks are in flight before conv4 starts
// (0.403 -> 0.385 ms per launch).
#pragma once
#include "gemm_pair_sm100.cuh"

namespace lrn {

struct ChainParams {
  int M;              // points covered by this launch
  int num_tiles;      // ceil(M / 256)
  const float4* ctx;  // (M) raw points [x, y, z, intensity]
  const float* w1;    // (64, 4) folded conv1, fp32
  const float* b1;    // (64)
  const float* wg1;   // (64) gate layer 1
  const float* bg1;   // (64)
  const float* b2;    // (128) folded biases of conv2..conv4
  const float* b3;    // (256)
  const float* b4;    // (512)
  const float* b5;    // (1024)
  void* cat;          // operand matrix (M, 2048) bf16 in the tiled layout (tmCat is its 4-D map: one store = one contiguous 16 KB block)
  long long* dbg;
};

constexpr int kChainStages = 3;
constexpr int kChainBlock = BM * 128;  // one [128 x 64] bf16 activation block / one weight stage: 16 KB

struct ChainSmem {
  static constexpr int kF1 = 0;                          // 1 block
  static constexpr int kF2 = kF1 + 1 * kChainBlock;      // 2 blocks; F2 + Z = 4 contiguous blocks = staging of feat4[0:256)
  static constexpr int kZ = kF2 + 2 * kChainBlock;       // 2 blocks
  static constexpr int kF3 = kZ + 2 * kChainBlock;       // 4 blocks; also staging of feat4[256:512) once conv4 has read it
  static constexpr int kGH = kF3 + 4 * kChainBlock;      // 1 block (gate hidden, staging for its TMA store only)
  static constexpr int kStages = kGH + 1 * kChainBlock;  // kChainStages weight stages of 16 KB
  static constexpr int kConst = kStages + kChainStages * kChainBlock;
  // fp32 constants: w1 (256) b1 (64) wg1 (64) bg1 (64) b2 (128) b3 (256) b4 (512) b5 (1024)
  static constexpr int kW1 = 0, kB1 = 256, kWg1 = 320, kBg1 = 384, kB2 = 448, kB3 = 576, kB4 = 832, kB5 = 1344,
                       kNumConst = 2368;
  // w_full[W] w_empty[W] act_ready[3] acc_full[2] acc_free[2] a4_ready acc5_full[2] acc5_free[2] fz_free x_full[2] f1gh_free f1gh_used
  static constexpr int kW = kChainStages + 4;  // + the four F2 / Z blocks borrowed as weight stages while conv5 runs
  static constexpr int kBarOff = kConst + kNumConst * 4;
  static constexpr int kTmemPtrOff = kBarOff + (2 * kW + 17) * 8;
  static constexpr int kTotal = kTmemPtrOff + 16;
  static constexpr int kDynamic = kTotal + 1024;
};

// Write 32 consecutive bf16 channels [c0, c0 + 32) of row `rr` into 64-column block(s) starting at `blocks`
// (block index c0 / 64), 128-byte swizzle: 16-byte piece c of a row sits at ((c ^ (row & 7)) << 4).
__device__ __forceinline__ void stage_packed_chunk(uint32_t blocks, int rr, int c0, const uint32_t* pk /* 16 */) {
  const uint32_t blk = blocks + (c0 >> 6) * kChainBlock + rr * 128;
  const int cbase = (c0 & 63) >> 3;
#pragma unroll
  for (int t = 0; t < 4; ++t)
    ptx::st_shared_v4(blk + (((cbase + t) ^ (rr & 7)) << 4), pk[4 * t], pk[4 * t + 1], pk[4 * t + 2], pk[4 * t + 3]);
}
// ... of relu(v): the clamp is part of the conversion (cvt.rn.relu.bf16x2)
__device__ __forceinline__ void stage_row_chunk_relu(uint32_t blocks, int rr, int c0, const float (&v)[32]) {
  uint32_t pk[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) pk[j] = ptx::pack_bf16x2_relu(v[2 * j], v[2 * j + 1]);
  stage_packed_chunk(blocks, rr, c0, pk);
}

// Drain NCHUNKS x 32 accumulator columns starting at TMEM address `t_addr` (layer column `col_lo`) of this
// thread's row: bias + ReLU -> bf16 -> swizzled smem blocks (the next layer's A operand and the TMA-store
// source).  TMEM loads are double-buffered.  chain_drain_keep also keeps the packed bf16 pairs in registers
// (they become a TMEM-resident A operand).
template <int NCHUNKS>
__device__ __forceinline__ void chain_drain_keep(uint32_t t_addr, int col_lo, const float* bias, uint32_t sblocks, int rr,
                                                 uint32_t (&keep)[NCHUNKS * 16]) {
  uint32_t r[2][32];
  ptx::tmem_ld_32x32b_x32(t_addr, r[0]);
#pragma unroll
  for (int i = 0; i < NCHUNKS; ++i) {
    const int c0 = col_lo + 32 * i;
    ptx::tmem_ld_wait();
    if (i + 1 < NCHUNKS) ptx::tmem_ld_32x32b_x32(t_addr + 32 * (i + 1), r[(i + 1) & 1]);
#pragma unroll
    for (int j = 0; j < 16; ++j)
      keep[16 * i + j] = ptx::pack_bf16x2_relu(__uint_as_float(r[i & 1][2 * j]) + bias[c0 + 2 * j],
                                               __uint_as_float(r[i & 1][2 * j + 1]) + bias[c0 + 2 * j + 1]);
    stage_packed_chunk(sblocks, rr, c0, &keep[16 * i]);
  }
}

template <int NCHUNKS>
__device__ __forceinline__ void chain_drain(uint32_t t_addr, int col_lo, const float* bias, uint32_t sblocks, int rr) {
  uint32_t r[2][32];
  ptx::tmem_ld_32x32b_x32(t_addr, r[0]);
#pragma unroll
  for (int i = 0; i < NCHUNKS; ++i) {
    const int c0 = col_lo + 32 * i;
    ptx::tmem_ld_wait();
    if (i + 1 < NCHUNKS) ptx::tmem_ld_32x32b_x32(t_addr + 32 * (i + 1), r[(i + 1) & 1]);
    uint32_t pk[16];   // bias + ReLU + bf16 rounding: one FADD per value, one cvt.rn.relu.bf16x2 per pair
#pragma unroll
    for (int j = 0; j < 16; ++j)
      pk[j] = ptx::pack_bf16x2_relu(__uint_as_float(r[i & 1][2 * j]) + bias[c0 + 2 * j], __uint_as_float(r[i & 1][2 * j + 1]) + bias[c0 + 2 * j + 1]);
    stage_packed_chunk(sblocks, rr, c0, pk);
  }
}

// 256 x N x 16 MMA over a CTA pair with the A operand in tensor memory (each CTA: its own 128 rows).
__device__ __forceinline__ void tc_mma_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
chain_pair_kernel(const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmW3,
                  const __grid_constant__ CUtensorMap tmW4, const __grid_constant__ CUtensorMap tmW5,
                  const __grid_constant__ CUtensorMap tmCat, const ChainParams p) {
  using L = ChainSmem;
  constexpr int S = kChainStages;
  constexpr uint32_t kIdesc128 = ptx::make_idesc(false, 2 * BM, 128);
  constexpr uint32_t kIdesc256 = ptx::make_idesc(false, 2 * BM, 256);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  float* sconst = reinterpret_cast<float*>(smem + L::kConst);
  constexpr int W = L::kW;
  uint64_t* w_full = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* w_empty = w_full + W;
  uint64_t* act_ready = w_empty + W;  // [3]: F1 / F2 / F3 of BOTH CTAs written (leader's copy is used)
  uint64_t* acc_full = act_ready + 3;  // [2]: accumulator buffer written by the MMAs
  uint64_t* acc_free = acc_full + 2;   // [2]: accumulator buffer drained by both CTAs (leader's copy is used)
  uint64_t* a4_ready = acc_free + 2;   // feat4 of BOTH CTAs is in tensor memory (leader's copy is used)
  uint64_t* acc5_full = a4_ready + 1;  // [2]: conv5 accumulator chunk written
  uint64_t* acc5_free = acc5_full + 2; // [2]: conv5 accumulator chunk drained by both CTAs (leader's copy is used)
  uint64_t* fz_free = acc5_free + 2;   // this CTA's F2 / Z blocks may be overwritten by conv5 weights (local)
  // The first two weight stages of a tile's conv5 (chunk 0, K = 0..255) live in the F1 / GH blocks, which are idle from
  // the end of conv2 until the next tile's conv1: those loads are issued ~10k cycles before feat4 is complete, so conv5
  // starts with its weights in place instead of waiting a TMA round trip for them (2k cycles per tile).
  uint64_t* x_full = fz_free + 1;      // [2]: weights landed in F1 / GH (both CTAs' halves; leader's copy is used)
  uint64_t* f1gh_free = x_full + 2;    // this CTA's F1 / GH: conv2 has read F1, their TMA store has been read (local)
  uint64_t* f1gh_used = f1gh_free + 1; // conv5's MMAs on the F1 / GH weights have completed (both CTAs, by tcgen05.commit)
  // weight stage s: 0..S-1 = dedicated stages, S..S+3 = blocks F2[0], F2[1], Z[0], Z[1]
  auto stage_ptr = [&](int st) { return smem + (st < S ? L::kStages + st * kChainBlock : L::kF2 + (st - S) * kChainBlock); };
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::kTmemPtrOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  // Once every CTA of this grid (at most one per SM) runs, the fusion kernel behind it may be launched: its CTAs
  // take over the SMs one by one as this grid's CTAs exit and wait in griddepcontrol.wait before their first operand load.
  ptx::launch_dependents();

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmW2);
    ptx::prefetch_tmap(&tmW3);
    ptx::prefetch_tmap(&tmW4);
    ptx::prefetch_tmap(&tmW5);
    ptx::prefetch_tmap(&tmCat);
    for (int s = 0; s < W; ++s) {
      ptx::mbar_init(&w_full[s], 1);
      ptx::mbar_init(&w_empty[s], 1);
    }
    ptx::mbar_init(fz_free, 1);
    ptx::mbar_init(&x_full[0], 1);
    ptx::mbar_init(&x_full[1], 1);
    ptx::mbar_init(f1gh_free, 1);
    ptx::mbar_init(f1gh_used, 1);
    for (int i = 0; i < 3; ++i) ptx::mbar_init(&act_ready[i], 2 * kPairEpiWarps);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&acc_free[i], 2 * kPairEpiWarps);
      ptx::mbar_init(&acc5_full[i], 1);
      ptx::mbar_init(&acc5_free[i], 2 * kPairEpiWarps);
    }
    ptx::mbar_init(a4_ready, 2 * kPairEpiWarps);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc_pair<512>(tmem_ptr);
  if (warp >= 2) {  // layer constants -> shared memory, once
    const int t = threadIdx.x - 64;
    for (int i = t; i < L::kNumConst; i += 32 * kPairEpiWarps) {
      float v;
      if (i < L::kB1) v = p.w1[i];
      else if (i < L::kWg1) v = p.b1[i - L::kB1];
      else if (i < L::kBg1) v = p.wg1[i - L::kWg1];
      else if (i < L::kB2) v = p.bg1[i - L::kBg1];
      else if (i < L::kB3) v = p.b2[i - L::kB2];
      else if (i < L::kB4) v = p.b3[i - L::kB3];
      else if (i < L::kB5) v = p.b4[i - L::kB4];
      else v = p.b5[i - L::kB5];
      sconst[i] = v;
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // one [128 rows x 64 columns] activation block -> operand matrix (row0 is a multiple of 128, col of 64)
  auto store_blk = [&](const void* smem_src, int col, int row0) {
    ptx::tma_store_4d(&tmCat, smem_src, 0, 0, col >> 6, row0 >> 7);
  };

  // Producer and MMA issue loops run warp-converged with the TMA / tcgen05 instructions predicated on elect.sync
  // (uniform-register operands, no per-lane serialisation), and the MMA loop looks at the next weight stage's barrier
  // while the current k-block is being issued: see gemm_pair_sm100.cuh and tools/mma_probe.cu.
  if (warp == 0) {
    // ------------------------------------------------------------ weight producer (both CTAs)
    // Two stage sequences share the per-stage barriers: conv2..conv4 cycle over the S dedicated stages (pointer
    // pa), conv5 over all W stages (pointer pb).  Parities are tracked per stage (bit s of `par`); the MMA warp
    // walks the identical sequence.
    int pa = 0, pb = 0, it = 0;
    uint32_t par = 0;
    const uint32_t full_leader0 = ptx::mapa(ptx::smem_u32(&w_full[0]), 0);
    auto load = [&](int st, const CUtensorMap* tm, int kcol, int nrow, uint32_t bytes) {
      ptx::mbar_wait(&w_empty[st], ((par >> st) & 1) ^ 1);
      par ^= 1u << st;
      if (ptx::elect_one()) {
        if (leader) ptx::mbar_arrive_expect_tx(&w_full[st], 2 * bytes);
        ptx::tma_load_2d_pair(stage_ptr(st), tm, full_leader0 + 8u * st, kcol, nrow);
      }
      __syncwarp();
    };
    auto next_a = [&]() { const int st = pa; pa = pa + 1 == S ? 0 : pa + 1; return st; };
    for (int tile = cluster_id; tile < p.num_tiles; tile += num_clusters, ++it) {
      load(next_a(), &tmW2, 0, static_cast<int>(rank) * 64, 64 * 128);                                    // conv2: N = 128
      for (int kb = 0; kb < 2; ++kb) load(next_a(), &tmW3, kb * 64, static_cast<int>(rank) * 128, 128 * 128);  // conv3: N = 256
      // conv4: 2 x (N = 256), eight 16 KB k-blocks per CTA.  Three dedicated stages cannot cover a ~2.8k-cycle TMA round trip
      // at conv4's rate (a k-block is consumed in ~0.5k cycles): the second and third k-block of the first chunk land in the
      // two Z blocks, which are idle from the end of the previous tile's conv5 until this tile's first conv4 drain stages
      // feat4 through them (that drain waits for the whole chunk's MMAs) - five k-blocks are in flight before conv4 starts.
      for (int c = 0; c < 2; ++c)
        for (int kb = 0; kb < 4; ++kb)
          load((c == 0 && (kb == 1 || kb == 2)) ? S + 1 + kb : next_a(), &tmW4, kb * 64, c * 256 + static_cast<int>(rank) * 128, 128 * 128);
      {                                                                                                  // conv5: 8 x (N = 128)
        bool fz_ok = false;
        for (int n = 0; n < 8; ++n)
          for (int kb2 = 0; kb2 < 4; ++kb2) {   // one stage = two 64-wide k-blocks of this CTA's 64 weight rows (2 x 8 KB)
            if (n == 0 && kb2 < 2) {  // the tile's first two conv5 stages: F1 / GH, free long before feat4 is complete
              if (kb2 == 0) ptx::mbar_wait(f1gh_free, it & 1);
              if (ptx::elect_one()) {
                uint8_t* dst = smem + (kb2 == 0 ? L::kF1 : L::kGH);
                const uint32_t xl = ptx::mapa(ptx::smem_u32(&x_full[kb2]), 0);
                if (leader) ptx::mbar_arrive_expect_tx(&x_full[kb2], 2 * kChainBlock);
                const int nrow = static_cast<int>(rank) * 64;
                ptx::tma_load_2d_pair(dst, &tmW5, xl, (2 * kb2) * 64, nrow);
                ptx::tma_load_2d_pair(dst + kChainBlock / 2, &tmW5, xl, (2 * kb2 + 1) * 64, nrow);
              }
              __syncwarp();
              continue;
            }
            const int st = pb;
            pb = pb + 1 == W ? 0 : pb + 1;
            if (st >= S && !fz_ok) {  // borrowed block: the feat4 store that staged through it must have drained it
              ptx::mbar_wait(fz_free, it & 1);
              fz_ok = true;
            }
            ptx::mbar_wait(&w_empty[st], ((par >> st) & 1) ^ 1);
            par ^= 1u << st;
            if (ptx::elect_one()) {
              if (leader) ptx::mbar_arrive_expect_tx(&w_full[st], 2 * kChainBlock);
              const int nrow = n * 128 + static_cast<int>(rank) * 64;
              ptx::tma_load_2d_pair(stage_ptr(st), &tmW5, full_leader0 + 8u * st, (2 * kb2) * 64, nrow);
              ptx::tma_load_2d_pair(stage_ptr(st) + kChainBlock / 2, &tmW5, full_leader0 + 8u * st, (2 * kb2 + 1) * 64, nrow);
            }
            __syncwarp();
          }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA)
    if (leader) {
      int pa = 0, pb = 0, it = 0;
      uint32_t wpar = 0;  // per-stage parity of w_full (same stage sequence as the producer)
      int peek_st = -1;   // stage whose full barrier was already seen complete while the previous k-block was issued
      // wait for weight stage `st` (unless the look-ahead has seen it), then look at stage `nx` (the next one of the same sequence)
      auto wait_stage = [&](int st, int nx) {
        if (peek_st != st) ptx::mbar_wait(&w_full[st], (wpar >> st) & 1);
        wpar ^= 1u << st;
        ptx::tc_fence_after();
        peek_st = ptx::mbar_test_wait(&w_full[nx], (wpar >> nx) & 1) ? nx : -1;
      };
      // one weight k-block: A = activation block `a_off` of this CTA (and the peer's at the same offset)
      auto kblock = [&](uint32_t a_off, uint32_t d_tmem, uint32_t idesc, bool first) {
        const int st = pa;
        pa = pa + 1 == S ? 0 : pa + 1;
        wait_stage(st, pa);
        if (ptx::elect_one()) {
          const uint64_t da = ptx::make_smem_desc_sw128(ptx::smem_u32(smem + a_off));
          const uint64_t db = ptx::make_smem_desc_sw128(ptx::smem_u32(stage_ptr(st)));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::tc_mma_ss_pair<false>(d_tmem, da + 2 * k, db + 2 * k, idesc, (!first || k > 0) ? 1u : 0u);
          ptx::tc_commit_pair(&w_empty[st], 3);
        }
        __syncwarp();
      };
      // the same for an explicit stage `st` (next stage of the sequence: `nx`)
      auto kblock_at = [&](int st, int nx, uint32_t a_off, uint32_t d_tmem, uint32_t idesc, bool first) {
        wait_stage(st, nx);
        if (ptx::elect_one()) {
          const uint64_t da = ptx::make_smem_desc_sw128(ptx::smem_u32(smem + a_off));
          const uint64_t db = ptx::make_smem_desc_sw128(ptx::smem_u32(stage_ptr(st)));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::tc_mma_ss_pair<false>(d_tmem, da + 2 * k, db + 2 * k, idesc, (!first || k > 0) ? 1u : 0u);
          ptx::tc_commit_pair(&w_empty[st], 3);
        }
        __syncwarp();
      };
      auto commit_acc = [&](int buf) {
        if (ptx::elect_one()) ptx::tc_commit_pair(&acc_full[buf], 3);
        __syncwarp();
      };
      for (int tile = cluster_id; tile < p.num_tiles; tile += num_clusters, ++it) {
        const uint32_t par = it & 1;
        const bool stamp = p.dbg && cluster_id == 0 && lane == 0 && it < 16;
        LRN_STAMP(stamp, p.dbg, it * 8 + 0);
        // Barrier bookkeeping.  The conv4 chunks are not handed back through acc_free (buf0 becomes conv5's A operand,
        // buf1 its accumulators): acc_free completes once per tile, and the buffers are reusable once the tensor pipe
        // (in order) is past conv5 and acc5_free says the last conv5 chunks have been drained.
        // conv2: F1 (K = 64) -> buf0[0:128)
        ptx::mbar_wait(&act_ready[0], par);
        ptx::tc_fence_after();
        kblock(L::kF1, tmem_base, kIdesc128, true);
        commit_acc(0);
        // conv3: F2 (K = 128) -> buf1
        ptx::mbar_wait(&act_ready[1], par);
        ptx::mbar_wait(&acc5_free[0], 1);  // previous tile's last two conv5 chunks drained (four completions per
        ptx::mbar_wait(&acc5_free[1], 1);  // buffer and tile: the phase parity is back to 0)
        ptx::tc_fence_after();
        for (int kb = 0; kb < 2; ++kb) kblock(L::kF2 + kb * kChainBlock, tmem_base + 256, kIdesc256, kb == 0);
        commit_acc(1);
        // conv4: F3 (K = 256) -> buf0 (channels 0..255), buf1 (channels 256..511)
        ptx::mbar_wait(&act_ready[2], par);
        {
          int stq[9];   // weight stages in the producer's order: k-blocks 1 and 2 of the first chunk sit in the Z blocks
          for (int i = 0; i < 8; ++i) {
            if (i == 1 || i == 2) {
              stq[i] = S + 1 + i;
            } else {
              stq[i] = pa;
              pa = pa + 1 == S ? 0 : pa + 1;
            }
          }
          stq[8] = pa;
          for (int c = 0; c < 2; ++c) {
            ptx::mbar_wait(&acc_free[c], par);  // this tile's conv2 / conv3 accumulator drained
            ptx::tc_fence_after();
            for (int kb = 0; kb < 4; ++kb)
              kblock_at(stq[4 * c + kb], stq[4 * c + kb + 1], L::kF3 + kb * kChainBlock, tmem_base + c * 256, kIdesc256, kb == 0);
            commit_acc(c);
          }
        }
        {
          // conv5: A = feat4 in TMEM columns [0, 256) (K = 512); eight 128-channel chunks alternate between two
          // accumulators (columns [256, 384) and [384, 512)), so chunk n + 1 runs while chunk n is drained.
          ptx::mbar_wait(a4_ready, par);
          ptx::tc_fence_after();
          const bool stamp5 = p.dbg && cluster_id == 0 && lane == 0 && it == 1;
          LRN_STAMP(stamp5, p.dbg, 128 + 8);  // feat4 in TMEM
          for (int n = 0; n < 8; ++n) {
            const int b = n & 1, j = n >> 1;
            ptx::mbar_wait(&acc5_free[b], (j & 1) ^ 1);  // chunk n - 2 (or the previous tile's chunk 6 / 7) drained
            ptx::tc_fence_after();
            LRN_STAMP(stamp5, p.dbg, 128 + 16 + n);  // accumulator free
            for (int kb2 = 0; kb2 < 4; ++kb2) {
              if (n == 0 && kb2 < 2) {  // weights of the tile's first two conv5 stages sit in F1 / GH
                ptx::mbar_wait(&x_full[kb2], par);
                ptx::tc_fence_after();
                if (ptx::elect_one()) {
                  const uint32_t wb = ptx::smem_u32(smem + (kb2 == 0 ? L::kF1 : L::kGH));
#pragma unroll
                  for (int h = 0; h < 2; ++h) {
                    const uint64_t db = ptx::make_smem_desc_sw128(wb + h * (kChainBlock / 2));
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                      tc_mma_ts_pair(tmem_base + 256, tmem_base + (2 * kb2 + h) * 32 + k * 8, db + 2 * k, kIdesc128,
                                     (kb2 > 0 || h > 0 || k > 0) ? 1u : 0u);
                  }
                  if (kb2 == 1) ptx::tc_commit_pair(f1gh_used, 3);   // F1 / GH may take the next tile's conv1 output
                }
                __syncwarp();
                continue;
              }
              const int st = pb;
              pb = pb + 1 == W ? 0 : pb + 1;
              wait_stage(st, pb);
              if (ptx::elect_one()) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  const uint64_t db = ptx::make_smem_desc_sw128(ptx::smem_u32(stage_ptr(st)) + h * (kChainBlock / 2));
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    tc_mma_ts_pair(tmem_base + 256 + 128 * b, tmem_base + (2 * kb2 + h) * 32 + k * 8, db + 2 * k, kIdesc128,
                                   (kb2 > 0 || h > 0 || k > 0) ? 1u : 0u);
                }
                ptx::tc_commit_pair(&w_empty[st], 3);
                if (kb2 == 3) ptx::tc_commit_pair(&acc5_full[b], 3);
              }
              __syncwarp();
            }
            LRN_STAMP(stamp5, p.dbg, 128 + n);  // chunk n issued
          }
        }
        LRN_STAMP(stamp, p.dbg, it * 8 + 1);
      }
    }
  } else {
    // ------------------------------------------------------------ compute / epilogue warps (both CTAs)
    const int ew = warp - 2;
    const int q = warp & 3;
    const int sub = ew >> 2;
    const int rr = q * 32 + lane;  // row (point) of this thread inside the CTA's 128
    const bool issuer = ew == 0 && lane == 0;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t sF1 = ptx::smem_u32(smem + L::kF1), sF2 = ptx::smem_u32(smem + L::kF2);
    const uint32_t sF3 = ptx::smem_u32(smem + L::kF3), sGH = ptx::smem_u32(smem + L::kGH);
    const uint32_t ready_leader0 = ptx::mapa(ptx::smem_u32(&act_ready[0]), 0);
    const uint32_t free_leader0 = ptx::mapa(ptx::smem_u32(&acc_free[0]), 0);

    // Before a block is rewritten, the TMA store that last read it must have finished reading shared memory.
    // Store groups are committed in program order  F2(t) F3(t) F1GH(t+1) f4c0(t) f4c1(t) F2(t+1) ...; `keep` =
    // number of groups committed AFTER the one that must be complete (they may stay in flight).
    auto staging_free = [&](int keep) {
      if (issuer) {
        if (keep >= 4) ptx::bulk_wait_read_keep<4>();
        else if (keep == 3) ptx::bulk_wait_read_keep<3>();
        else if (keep == 2) ptx::bulk_wait_read_keep<2>();
        else if (keep == 1) ptx::bulk_wait_read_keep<1>();
        else ptx::bulk_wait_read_all();
      }
      ptx::named_bar_sync(1, 32 * kPairEpiWarps);
    };
    // conv1 and gate layer 1 for one tile: raw point -> 64 + 64 bf16 channels of blocks F1 / GH (each warp group: half of both)
    // this thread's raw point of a tile (requested a whole tile ahead: a DRAM round trip is ~1k cycles)
    auto load_point = [&](int tile) {
      const int grow = tile * 2 * BM + static_cast<int>(rank) * BM + rr;
      return tile < p.num_tiles && grow < p.M ? __ldg(p.ctx + grow) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    // The work is split in two steps (conv1 -> F1, gate layer 1 -> GH + hand-over) so that, done between conv5 chunk
    // drains, neither step is longer than the slack the double-buffered conv5 accumulators can absorb.
    auto embed = [&](int tile, const float4 x, int part /* 0: conv1, 1: gate + hand-over, 2: both */) {
      const int row0 = tile * 2 * BM + static_cast<int>(rank) * BM;
      if (part != 1) staging_free(4);  // the F1GH store of the previous use of these blocks lies many groups back
      {
        // both warp groups do half of each: channels [32 sub, 32 sub + 32) of conv1 (4 FMA per channel) and of the gate's
        // first layer (1 FMA per channel) - conv1 on one group and the gate on the other left the conv1 warps 4x longer
        const int h = sub;
        float v[32];
        if (part != 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float4 w = reinterpret_cast<const float4*>(sconst + L::kW1)[32 * h + j];
            v[j] = fmaf(w.x, x.x, fmaf(w.y, x.y, fmaf(w.z, x.z, fmaf(w.w, x.w, sconst[L::kB1 + 32 * h + j]))));
          }
          stage_row_chunk_relu(sF1, rr, 32 * h, v);
          if (part == 0) return;
        }
#pragma unroll
        for (int j = 0; j < 32; ++j)
          v[j] = fmaf(sconst[L::kWg1 + 32 * h + j], x.w, sconst[L::kBg1 + 32 * h + j]);
        stage_row_chunk_relu(sGH, rr, 32 * h, v);
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(ready_leader0);
      ptx::named_bar_sync(1, 32 * kPairEpiWarps);
      if (issuer) {
        // The first store into the operand matrix waits for the kernel this one was launched behind (the previous
        // wave's fusion kernel reads the same buffer); everything up to here - setup, weight loads, the first tile's
        // points, conv1 / gate layer 1, and conv2 on the tensor pipe - overlaps that kernel's last tiles.
        if (tile == cluster_id) ptx::grid_dependency_wait();
        store_blk(smem + L::kF1, 0, row0);
        store_blk(smem + L::kGH, 1984, row0);
        ptx::bulk_commit();
      }
    };

    int it = 0;
    if (cluster_id < p.num_tiles) embed(cluster_id, load_point(cluster_id), 2);
    for (int tile = cluster_id; tile < p.num_tiles; tile += num_clusters, ++it) {
      const int row0 = tile * 2 * BM + static_cast<int>(rank) * BM;
      const float4 x_next = load_point(tile + num_clusters);
      // ---- conv2 epilogue: buf0[0:128) -> F2 (2 blocks); this warp: columns [64 sub, 64 sub + 64)
      const bool stamp = p.dbg && cluster_id == 0 && leader && warp == 2 && lane == 0 && it < 16;
      // F2 doubled as staging in the previous tile (feat4 chunk 0) and every group up to the last one committed has been
      // read; on the first tile the only group is F1GH of this very tile, which must be complete before F1 / GH are reused
      staging_free(it == 0 ? 0 : 1);
      ptx::mbar_wait(&acc_full[0], 0);
      ptx::tc_fence_after();
      if (issuer) ptx::mbar_arrive(f1gh_free);  // conv2 has read F1, the F1GH store has been read: conv5 weights may land there
      LRN_STAMP(stamp, p.dbg, it * 8 + 2);  // conv2 accumulator ready
      chain_drain<2>(t_lane + 64 * sub, 64 * sub, sconst + L::kB2, sF2, rr);
      ptx::tc_fence_before();
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive_cluster(free_leader0);       // buf0 drained
        ptx::mbar_arrive_cluster(ready_leader0 + 8);  // F2 written
      }
      ptx::named_bar_sync(1, 32 * kPairEpiWarps);
      if (issuer) {
        store_blk(smem + L::kF2, 64, row0);
        store_blk(smem + L::kF2 + kChainBlock, 128, row0);
        ptx::bulk_commit();
      }
      LRN_STAMP(stamp, p.dbg, it * 8 + 3);  // conv2 drained, F2 stores issued
      // ---- conv3 epilogue: buf1 -> F3 (4 blocks); this warp: columns [128 sub, 128 sub + 128)
      staging_free(1);  // F3 doubled as feat4 staging of the previous tile: f4c1(t-1), then only F2(t)
      ptx::mbar_wait(&acc_full[1], 0);
      ptx::tc_fence_after();
      LRN_STAMP(stamp, p.dbg, it * 8 + 4);  // conv3 accumulator ready
      chain_drain<4>(t_lane + 256 + 128 * sub, 128 * sub, sconst + L::kB3, sF3, rr);
      ptx::tc_fence_before();
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive_cluster(free_leader0 + 8);    // buf1 drained
        ptx::mbar_arrive_cluster(ready_leader0 + 16);  // F3 written
      }
      ptx::named_bar_sync(1, 32 * kPairEpiWarps);
      if (issuer) {
#pragma unroll
        for (int b = 0; b < 4; ++b) store_blk(smem + L::kF3 + b * kChainBlock, 192 + 64 * b, row0);
        ptx::bulk_commit();
      }
      LRN_STAMP(stamp, p.dbg, it * 8 + 5);  // conv3 drained, F3 stores issued
      const bool has_next = tile + num_clusters < p.num_tiles;
      LRN_STAMP(stamp, p.dbg, it * 8 + 6);
      // ---- conv4 epilogues: feat4 channels [256 c + 128 sub, +128) -> staging blocks -> operand row columns 448 + ...
      //      chunk 0 is staged in F2 + Z (conv3 of this tile is done with F2), chunk 1 in F3 (all of conv4 has
      //      completed once its accumulator is ready).
      for (int c = 0; c < 2; ++c) {
        // c = 0 needs F2(t) drained (later group: F3(t)); c = 1 needs F3(t) (later group: f4c0(t))
        staging_free(1);
        ptx::mbar_wait(&acc_full[c], 1);
        ptx::tc_fence_after();
        uint32_t keep[64];
        if (c == 0) {
          chain_drain_keep<4>(t_lane + 128 * sub, 128 * sub, sconst + L::kB4, sF2, rr, keep);
        } else {
          // Drain in two halves: in between, feat4 chunk 0's store (staged in F2 + Z, committed at the end of the c = 0
          // pass) has long been read, so the issuer can hand those four blocks to the weight producer NOW - conv5's
          // borrowed weight stages are then in flight ~1.5k cycles before feat4 is complete instead of after it (the
          // first conv5 chunk used to wait ~2.9k cycles for its fourth weight stage).
          uint32_t (&lo)[32] = reinterpret_cast<uint32_t(&)[32]>(keep[0]);
          uint32_t (&hi)[32] = reinterpret_cast<uint32_t(&)[32]>(keep[32]);
          chain_drain_keep<2>(t_lane + 256 + 128 * sub, 128 * sub, sconst + L::kB4 + 256, sF3, rr, lo);
          if (issuer) {
            ptx::bulk_wait_read_all();
            ptx::mbar_arrive(fz_free);
          }
          chain_drain_keep<2>(t_lane + 256 + 128 * sub + 64, 128 * sub + 64, sconst + L::kB4 + 256, sF3, rr, hi);
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        __syncwarp();
        ptx::named_bar_sync(1, 32 * kPairEpiWarps);  // every warp is done reading this accumulator buffer
        if (issuer) {
#pragma unroll
          for (int b = 0; b < 4; ++b)
            store_blk(smem + (c == 0 ? L::kF2 : L::kF3) + b * kChainBlock, 448 + 256 * c + 64 * b, row0);
          ptx::bulk_commit();
        }
        {
          // feat4 channels [256 c + 128 sub, +128) as conv5's A operand: packed columns [128 c + 64 sub, +64) of buf0
          // (all reads of buf0 by chunk 0 finished at the barrier above / one iteration earlier)
          ptx::tc_fence_after();
          ptx::tmem_st_32x32b_x32(t_lane + 128 * c + 64 * sub, reinterpret_cast<const uint32_t(&)[32]>(keep[0]));
          ptx::tmem_st_32x32b_x32(t_lane + 128 * c + 64 * sub + 32, reinterpret_cast<const uint32_t(&)[32]>(keep[32]));
          ptx::tmem_st_wait();
          if (c == 1) {
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(a4_ready), 0));
          }
        }
      }
      {
        // ---- conv5 epilogues: chunk n = channels [128 n, +128) in accumulator n & 1; this warp: columns [64 sub, +64)
        //      -> staging blocks F3[2 (n & 1) + sub] (F2 / Z hold conv5 weights now) -> operand row columns 960 + 128 n + 64 b
        const uint32_t free5_leader0 = ptx::mapa(ptx::smem_u32(&acc5_free[0]), 0);
        for (int n = 0; n < 8; ++n) {
          const int b = n & 1, j = n >> 1;
          // blocks 2b, 2b + 1 of F3 were last read by the store of feat4 chunk 1 (n < 2) or of conv5 chunk n - 2: everything
          // but the most recent group (chunk n - 1) must have been read - and, for n = 4, 5, the F1GH group of the next
          // tile's conv1 / gate layer 1, which is committed between chunks 3 and 4
          staging_free(n == 0 ? 0 : ((n == 4 || n == 5) && has_next) ? 2 : 1);
          const bool stamp5 = p.dbg && cluster_id == 0 && leader && warp == 2 && lane == 0 && it == 1;
          LRN_STAMP(stamp5, p.dbg, 128 + 24 + n);  // staging free
          ptx::mbar_wait(&acc5_full[b], j & 1);
          ptx::tc_fence_after();
          LRN_STAMP(stamp5, p.dbg, 128 + 32 + n);  // accumulator ready
          chain_drain<2>(t_lane + 256 + 128 * b + 64 * sub, 64 * sub, sconst + L::kB5 + 128 * n, sF3 + 2 * b * kChainBlock, rr);
          ptx::tc_fence_before();
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(free5_leader0 + 8 * b);
          ptx::named_bar_sync(1, 32 * kPairEpiWarps);
          if (issuer) {
#pragma unroll
            for (int bb = 0; bb < 2; ++bb)
              store_blk(smem + L::kF3 + (2 * b + bb) * kChainBlock, 960 + 128 * n + 64 * bb, row0);
            ptx::bulk_commit();
          }
          LRN_STAMP(stamp5, p.dbg, 128 + 40 + n);  // drained, stores issued
          if (has_next && (n == 1 || n == 3)) {
            // ---- next tile's conv1 (after chunk 1) and gate layer 1 (after chunk 3), in the shadow of conv5 (the epilogue
            //      warps idle about half of every chunk): F1 / GH held this tile's first conv5 weights until the tensor
            //      pipe finished the MMAs that read them
            if (n == 1) ptx::mbar_wait(f1gh_used, it & 1);
            embed(tile + num_clusters, x_next, n == 1 ? 0 : 1);
          }
        }
      }
      LRN_STAMP(stamp, p.dbg, it * 8 + 7);  // conv4 drained
    }
    if (issuer) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair<512>(tmem_base);
  }
}

}  // namespace lrn
