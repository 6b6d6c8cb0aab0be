// CTA-pair (cta_group::2) variant of the shared-MLP GEMM: one 256-point x BN-channel tile per
// cluster of two CTAs.  Each CTA stages its own 128 rows of A and HALF of the weight tile, the
// leader CTA's elected thread issues tcgen05.mma.cta_group::2 (M = 256), and each CTA's TMEM holds
// the accumulator rows of its own 128 points.  Compared with the single-CTA 128x128 tile this
// halves the operand bytes each SM has to pull through TMA per MMA cycle.
//
//   warp 0      : TMA producer (both CTAs; bytes are counted on the LEADER's full barrier)
//   warp 1      : TMEM allocator (both CTAs) + MMA issuer (leader only)
//   warps 2..9  : epilogue; warp w owns TMEM lane quarter (w & 3) and column half ((w - 2) >> 2)
//
// EPI_ACT   : 2 accumulator stages of BN columns (epilogue of tile i overlaps the MMAs of tile i+1)
// EPI_FUSION: BN = 256; the 512 TMEM columns are two regions R0/R1 of 256 columns.  Tile t keeps its
//             fusion accumulator F_t in R[t&1] and its (short-lived) gate accumulator G_t in the other
//             region, which is the one F_{t-1} occupied:
//               MMA pipe : ... F_{t-1} k-blocks | F_t k-blocks 0..9 | G_t | F_t k-blocks 10..30 | F_{t+1} ...
//               epilogue : phase B_{t-1} (reads F_{t-1})  ->  phase A_t (G_t -> gamma in REGISTERS)  ->  phase B_t
//             Phase A turns G into gamma = 0.5 + 0.5*sigmoid(G + bg) and keeps it as 16-bit fixed point in 64
//             registers per thread (gamma is in [0.5, 1): its top 16 mantissa bits, error < 4e-6), which frees
//             the region again, so consecutive main loops run back to back and both epilogue phases hide
//             under the 31 fusion k-blocks of the next tile.
#pragma once
#include "gemm_common.cuh"

namespace lrn {

constexpr int kPairEpiWarps = 8;
constexpr int kPairThreads = 64 + 32 * kPairEpiWarps;  // 320
constexpr int kPoolRowStride = 36;                      // floats; 16-byte aligned rows, conflict-free both ways

// STAGED: bf16 outputs leave through shared memory ([128 x 64] blocks in the 128-byte-swizzled layout TMA
// and UMMA share) and one TMA store per block, instead of 16-byte pieces of 32 different rows per instruction.
template <int BN, int STAGES, bool POOL, bool STAGED = false>
struct PairSmem {
  static constexpr int kA = BM * kTileRowBytes;        // this CTA's 128 rows
  static constexpr int kB = (BN / 2) * kTileRowBytes;  // this CTA's half of the weight tile
  static constexpr int kStage = kA + kB;
  static constexpr int kTiles = STAGES * kStage;
  static constexpr int kBarOff = kTiles;  // full[STAGES], empty[STAGES], tfull[2], tempty[2]
  static constexpr int kTmemPtrOff = kBarOff + (2 * STAGES + 4) * 8;
  static constexpr int kBiasOff = kTmemPtrOff + 16;                                // float sbias[2][2 * BN]
  static constexpr int kPoolOff = (kBiasOff + 2 * 2 * BN * 4 + 15) / 16 * 16;      // per-warp 32 x 36 float scratch
  static constexpr int kStagingOff = (kPoolOff + (POOL ? kPairEpiWarps * 32 * kPoolRowStride * 4 : 0) + 1023) / 1024 * 1024;
  static constexpr int kStagingBlock = BM * 128;  // 128 rows x 64 bf16
  static constexpr int kTotal = kStagingOff + (STAGED ? (BN / 64) * kStagingBlock : 0);
  static constexpr int kDynamic = kTotal + 1024;
};

// max / sum over the 32 points of a warp for 32 channels through a padded shared-memory transpose:
// 8 STS.128 + 32 LDS per lane instead of 2 x 31 shuffles with selects.  Lane l returns channel l.
__device__ __forceinline__ void pool_chunk_smem(const float (&v)[32], float* scratch, int lane, float& mx, float& sm) {
  float4* row = reinterpret_cast<float4*>(scratch + lane * kPoolRowStride);
#pragma unroll
  for (int q = 0; q < 8; ++q) row[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  __syncwarp();
  mx = 0.f;
  sm = 0.f;
#pragma unroll
  for (int r = 0; r < 32; ++r) {
    const float x = scratch[r * kPoolRowStride + lane];
    mx = fmaxf(mx, x);
    sm += x;
  }
  __syncwarp();
}

// Position `s` of tile `it` in the fusion kernel's k-block sequence: the gate k-blocks come first for
// the first tile of a CTA pair and are spliced in after a third of the fusion k-blocks afterwards
// (by then phase B of the previous tile has released the region G is accumulated in).
struct KbSlot {
  bool gate;
  int kb;  // index within its own group (gate / fusion)
};
__device__ __forceinline__ int fusion_gate_pos(int it, int kb_main) { return it == 0 ? 0 : kb_main / 3; }
__device__ __forceinline__ KbSlot fusion_slot(int ins, int s, int kb_gate) {
  if (s < ins) return {false, s};
  if (s < ins + kb_gate) return {true, s - ins};
  return {false, s - kb_gate};
}

// gamma in [0.5, 1] <-> 16-bit fixed point (the top 16 mantissa bits of a float in [0.5, 1))
__device__ __forceinline__ uint32_t gamma_pack(float lo, float hi) {
  const uint32_t a = min(__float_as_uint(lo) + 64u, 0x3F7FFFFFu);
  const uint32_t b = min(__float_as_uint(hi) + 64u, 0x3F7FFFFFu);
  return ((a >> 7) & 0xFFFFu) | ((b << 9) & 0xFFFF0000u);
}
__device__ __forceinline__ float gamma_lo(uint32_t q) { return __uint_as_float(0x3F000000u | ((q & 0xFFFFu) << 7)); }
__device__ __forceinline__ float gamma_hi(uint32_t q) { return __uint_as_float(0x3F000000u | ((q >> 16) << 7)); }

// GENERAL = false is the common fusion case (no argmax, every warp's 32 points valid and inside one
// segment: N % 32 == 0); it drops the masked / 64-bit-key pooling paths and their registers.
// MN = true (bf16, EPI_ACT): both operands are MN-major, i.e. the GEMM is  D[M x N] = A^T B  with A stored (K, M) and
// B stored (K, N) row-major -- the weight-gradient shape dW = dU^T X (K = points) straight from the point-major
// activation / gradient buffers, no transposed copies.  TMA boxes are [64 k-rows x 64 m/n] (128-byte rows).
template <int BN, bool TF32, int EPI, int STAGES, bool GENERAL = true, bool STAGED = false, bool MN = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmOut, const GemmParams p) {
  static_assert(!STAGED || (EPI == EPI_ACT && !TF32), "staged TMA stores are implemented for bf16 EPI_ACT outputs");
  using L = PairSmem<BN, STAGES, EPI == EPI_FUSION, STAGED>;
  constexpr int BK = TF32 ? 32 : 64;
  constexpr int kMmaPerKb = 4;
  constexpr uint32_t kTmemCols = 2 * BN;
  static_assert(kTmemCols == 256 || kTmemCols == 512, "TMEM columns must be a power of two");
  static_assert(EPI != EPI_FUSION || BN == 256, "fusion epilogue is laid out for BN = 256");
  static_assert(!MN || (EPI == EPI_ACT && !TF32 && !STAGED), "MN-major operands: bf16 EPI_ACT only");
  constexpr uint32_t kIdesc = ptx::make_idesc(TF32, 2 * BM, BN, MN);
  constexpr int kHalfCols = BN / 2;  // columns handled by one epilogue warp
  constexpr int kChunks = kHalfCols / 32;
  // bf16 fusion + gate + pooling: launched with programmatic stream serialization behind the chain kernel that writes its
  // operand rows (lrn_abi.cu), and followed by the next wave's chain kernel, which overwrites them
  constexpr bool kPdl = EPI == EPI_FUSION && !TF32;

  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic on the __shared__ array (keeps the shared address space: LDS/STS)
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* bar_empty = bar_full + STAGES;
  uint64_t* bar_tfull = bar_empty + STAGES;  // accumulator stage / TMEM region written  (MMA -> epilogue)
  uint64_t* bar_tempty = bar_tfull + 2;      // accumulator stage / TMEM region consumed (epilogue -> MMA, leader's copy)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::kTmemPtrOff);
  float* sbias = reinterpret_cast<float*>(smem + L::kBiasOff);
  float* spool = reinterpret_cast<float*>(smem + L::kPoolOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  // m_tiles counts 256-row pair tiles here; split-K (EPI_ACT, fp32 output) multiplies the tile count: work
  // item w = split * (m_tiles * n_tiles) + output tile, each covering kb_per_split k-blocks
  const int splits = (EPI == EPI_ACT && p.k_splits > 1) ? p.k_splits : 1;
  const int out_tiles = p.m_tiles * p.n_tiles;
  const int num_tiles = out_tiles * splits;
  const int kb_all = p.kb_main + p.kb_gate;
  auto kb_begin = [&](int w) { return splits > 1 ? (w / out_tiles) * p.kb_per_split : 0; };
  auto kb_count = [&](int w) { return splits > 1 ? min(p.kb_per_split, kb_all - kb_begin(w)) : kb_all; };
  // the next wave's chain kernel may start on the SMs this grid's CTAs leave (its stores wait for this grid)
  if (kPdl) ptx::launch_dependents();

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&bar_full[s], 1);   // leader: its own arrive.expect_tx (bytes of both CTAs)
      ptx::mbar_init(&bar_empty[s], 1);  // one multicast tcgen05.commit
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&bar_tfull[s], 1);
      ptx::mbar_init(&bar_tempty[s], 2 * kPairEpiWarps);  // every epilogue warp of both CTAs (leader's copy is used)
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc_pair<kTmemCols>(tmem_ptr);
  ptx::tc_fence_before();
  ptx::cluster_sync();  // barrier inits + TMEM allocation visible in both CTAs before any remote traffic
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // Both issue loops below are executed by the WHOLE warp with only the TMA / tcgen05 instructions predicated on
  // elect.sync: every address and descriptor is then provably warp-uniform and lives in uniform registers.  Issued from
  // an `if (lane == 0)` region the same instructions are wrapped in per-lane serialisation loops with R2UR moves, and
  // since the tensor pipe queues only about one MMA ahead, that issue latency (plus the barrier round trip per k-block)
  // showed up as ~194 instead of 128 cycles per 256x256x16 MMA (tools/mma_probe.cu, profiles/r02_mma_probe*.txt).
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    const uint32_t full_leader0 = ptx::mapa(ptx::smem_u32(&bar_full[0]), 0);
    // Behind the chain kernel (kPdl), the weight halves of the first tile's first STAGES k-blocks are loaded before
    // griddepcontrol.wait, and their operand-row halves, which the chain kernel writes, after it.  Each stage's
    // expect_tx still counts both halves.
    int b_early = 0;
    if (kPdl) {
      if (cluster_id < num_tiles) {
        const int n_blk = (cluster_id % out_tiles) % p.n_tiles;
        b_early = min(STAGES, kb_count(cluster_id));
        for (int s = 0; s < b_early; ++s) {
          const KbSlot slot = fusion_slot(fusion_gate_pos(0, p.kb_main), s, p.kb_gate);
          const int kcol = slot.gate ? p.kb_main + slot.kb : slot.kb;
          if (ptx::elect_one()) {
            if (leader) ptx::mbar_arrive_expect_tx(&bar_full[s], 2 * L::kStage);
            ptx::tma_load_2d_pair(smem + s * L::kStage + L::kA, &tmB, full_leader0 + 8u * s, kcol * BK,
                                  n_blk * BN + static_cast<int>(rank) * (BN / 2));
          }
          __syncwarp();
        }
      }
      ptx::grid_dependency_wait();
    }
    for (int work = cluster_id; work < num_tiles; work += num_clusters, ++it) {
      const int tile = work % out_tiles;
      const int m_blk = tile / p.n_tiles;
      const int n_blk = tile - m_blk * p.n_tiles;
      const int kb_total = kb_count(work), kb0 = kb_begin(work);
      const int ins = fusion_gate_pos(it, p.kb_main);
      for (int s = 0; s < kb_total; ++s) {
        int kcol = kb0 + s;
        if (EPI == EPI_FUSION) {  // the gate k-blocks are the last columns of the operand row
          const KbSlot slot = fusion_slot(ins, s, p.kb_gate);
          kcol = slot.gate ? p.kb_main + slot.kb : slot.kb;
        }
        int a_extra = 0, b_extra = 0;
        if (TF32 && p.split3) {  // three passes over the same k-blocks: A_hi B_hi, A_lo B_hi, A_hi B_lo
          KbSlot slot{false, s};
          if (EPI == EPI_FUSION) slot = fusion_slot(ins, s, p.kb_gate);
          const int n1 = (slot.gate ? p.kb_gate : p.kb_main) / 3;
          const int pass = slot.kb / n1;
          kcol = (slot.gate ? p.kb_main / 3 : 0) + slot.kb - pass * n1;
          a_extra = pass == 1 ? p.a_lo_off : 0;
          b_extra = pass == 2 ? p.b_lo_off : 0;
        }
        const bool b_loaded = kPdl && it == 0 && s < b_early;
        ptx::mbar_wait(&bar_empty[stage], phase ^ 1);
        if (ptx::elect_one()) {
          uint8_t* sa = smem + stage * L::kStage;
          const uint32_t full_leader = full_leader0 + 8u * stage;
          if (leader && !b_loaded) ptx::mbar_arrive_expect_tx(&bar_full[stage], 2 * L::kStage);
          if (MN) {  // boxes of 64 k-rows x 64 m/n columns: this CTA's 128 m and BN/2 n
#pragma unroll
            for (int b = 0; b < 2; ++b)
              ptx::tma_load_2d_pair(sa + b * 8192, &tmA, full_leader, m_blk * 2 * BM + static_cast<int>(rank) * BM + 64 * b,
                                    kcol * BK);
#pragma unroll
            for (int b = 0; b < BN / 128; ++b)
              ptx::tma_load_2d_pair(sa + L::kA + b * 8192, &tmB, full_leader,
                                    n_blk * BN + static_cast<int>(rank) * (BN / 2) + 64 * b, kcol * BK);
          } else {
#ifdef LRN_TIMELINE   // tools/l2_ring_probe.py: read the operand rows of tile (m_blk mod ring) - an L2-resident stand-in
            const int a_blk = p.a_ring > 0 ? m_blk % p.a_ring : m_blk;
#else
            const int a_blk = m_blk;
#endif
            if (p.a_tiled)  // one contiguous 16 KB block: (column block, row tile) of the tiled operand matrix
              ptx::tma_load_4d_pair(sa, &tmA, full_leader, 0, 0, (p.a_col0 + kcol * BK) / BK, a_blk * 2 + static_cast<int>(rank));
            else
              ptx::tma_load_2d_pair(sa, &tmA, full_leader, p.a_col0 + kcol * BK + a_extra, m_blk * 2 * BM + static_cast<int>(rank) * BM);
            if (!b_loaded)
              ptx::tma_load_2d_pair(sa + L::kA, &tmB, full_leader, kcol * BK + b_extra, n_blk * BN + static_cast<int>(rank) * (BN / 2));
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      bool peeked = false;  // the full barrier of `stage` was already seen complete (looked at one k-block ahead)
      for (int work = cluster_id; work < num_tiles; work += num_clusters, ++it) {
        const int kb_total = kb_count(work);
        const bool stamp = p.dbg && cluster_id == 0 && lane == 0 && it < 16;
        LRN_STAMP(stamp, p.dbg, it * 8 + 0);  // tile start
        // EPI_ACT: accumulator stage it&1, completes every second tile.  EPI_FUSION: F_t lives in region
        // it&1 and G_t in the other one; every region is written exactly once per tile, so all
        // region barriers complete once per tile (parity it&1).
        const int rf = it & 1;
        const uint32_t par_free = (EPI == EPI_FUSION) ? ((it & 1) ^ 1) : (((it >> 1) & 1) ^ 1);
        const uint32_t acc_main = tmem_base + rf * BN;
        const uint32_t acc_gate = tmem_base + (rf ^ 1) * BN;
        const int ins = fusion_gate_pos(it, p.kb_main);
        const int kb_last = (EPI == EPI_FUSION ? p.kb_main : kb_total) - 1;
        for (int s = 0; s < kb_total; ++s) {
          KbSlot slot{false, s};
          if (EPI == EPI_FUSION) slot = fusion_slot(ins, s, p.kb_gate);
          if (slot.kb == 0) {  // first write into this region/stage: wait until the epilogue has drained it
            ptx::mbar_wait(&bar_tempty[slot.gate ? (rf ^ 1) : rf], par_free);
            ptx::tc_fence_after();
          }
          if (!peeked) ptx::mbar_wait(&bar_full[stage], phase);
          ptx::tc_fence_after();
          const int cur = stage;
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
          // look at the next stage now: the answer arrives while this k-block's MMAs are being issued
          peeked = ptx::mbar_test_wait(&bar_full[stage], phase);
          if (ptx::elect_one()) {
            const uint32_t a_addr = ptx::smem_u32(smem + cur * L::kStage);
            const uint64_t da = MN ? ptx::make_smem_desc_sw128_mn(a_addr, 8192) : ptx::make_smem_desc_sw128(a_addr);
            const uint64_t db = MN ? ptx::make_smem_desc_sw128_mn(a_addr + L::kA, 8192) : ptx::make_smem_desc_sw128(a_addr + L::kA);
            const uint32_t d = slot.gate ? acc_gate : acc_main;
            // K step of one MMA (16 bf16): 32 bytes along a K-major row, or 16 k-rows = 2048 bytes of an MN-major tile
            constexpr int kStep = MN ? (2048 >> 4) : 2;
#pragma unroll
            for (int k = 0; k < kMmaPerKb; ++k)
              ptx::tc_mma_ss_pair<TF32>(d, da + kStep * k, db + kStep * k, kIdesc, (slot.kb > 0 || k > 0) ? 1u : 0u);
            ptx::tc_commit_pair(&bar_empty[cur], 3);  // frees this smem stage in BOTH CTAs
            if (slot.gate && slot.kb == p.kb_gate - 1) ptx::tc_commit_pair(&bar_tfull[rf ^ 1], 3);  // G_t complete
            if (!slot.gate && slot.kb == kb_last) ptx::tc_commit_pair(&bar_tfull[rf], 3);           // F_t complete
          }
          __syncwarp();
        }
        LRN_STAMP(stamp, p.dbg, it * 8 + 1);  // last MMA of the tile issued
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 2..9, both CTAs)
    const int ew = warp - 2;
    const int q = warp & 3;      // TMEM lane quarter
    const int half = ew >> 2;    // which half of the BN columns
    const int et = threadIdx.x - 64;
    float* scratch = spool + ew * 32 * kPoolRowStride;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int col_lo = half * kHalfCols;
    int it = 0;
    for (int work = cluster_id; work < num_tiles; work += num_clusters, ++it) {
      const int tile = work % out_tiles;
      const int m_blk = tile / p.n_tiles;
      const int n_blk = tile - m_blk * p.n_tiles;
      const bool add_bias = work < out_tiles;  // split-K: only the first split adds the bias
      float* sb = sbias + (it & 1) * 2 * BN;
      for (int c = et; c < BN; c += 32 * kPairEpiWarps) {
        if (EPI == EPI_FUSION) {
          sb[c] = p.bias_f[n_blk * BN + c];
          sb[BN + c] = p.bias_g[n_blk * BN + c];
        } else {
          sb[c] = (p.bias && add_bias) ? p.bias[n_blk * BN + c] : 0.f;
        }
      }
      ptx::named_bar_sync(1, 32 * kPairEpiWarps);

      const int row = m_blk * 2 * BM + static_cast<int>(rank) * BM + q * 32 + lane;  // row within this launch
      const bool valid = row < p.M;

      if (EPI == EPI_ACT) {
        const int as = it & 1;
        uint8_t* staging = smem + L::kStagingOff;
        const bool issuer = (ew & 3) == 0 && lane == 0;  // one thread per column half issues the TMA stores
        const bool stamp = p.dbg && cluster_id == 0 && leader && warp == 2 && lane == 0 && it < 16;
        LRN_STAMP(stamp, p.dbg, it * 8 + 2);  // epilogue of this tile starts
        if (STAGED) {
          if (issuer) ptx::bulk_wait_read_all();  // the previous tile's stores have drained the staging blocks
          ptx::named_bar_sync(2 + half, 128);
        }
        LRN_STAMP(stamp, p.dbg, it * 8 + 3);  // staging free
        ptx::mbar_wait(&bar_tfull[as], (it >> 1) & 1);
        ptx::tc_fence_after();
        LRN_STAMP(stamp, p.dbg, it * 8 + 4);  // accumulator ready
        // software-pipelined: the TMEM load of chunk i+1 is in flight while chunk i is converted and stored
        uint32_t r[2][32];
        ptx::tmem_ld_32x32b_x32(t_lane + as * BN + col_lo, r[0]);
#pragma unroll
        for (int i = 0; i < kChunks; ++i) {
          const int c0 = col_lo + 32 * i;
          ptx::tmem_ld_wait();
          if (i + 1 < kChunks) ptx::tmem_ld_32x32b_x32(t_lane + as * BN + c0 + 32, r[(i + 1) & 1]);
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float x = __uint_as_float(r[i & 1][j]) + sb[c0 + j];
            v[j] = p.relu ? fmaxf(x, 0.f) : x;
          }
          if (STAGED) {
            // row r of block b: 128 bytes, 16-byte piece c lives at ((c ^ (r & 7)) << 4)  (128B swizzle)
            const int rr = q * 32 + lane;
            const uint32_t blk = ptx::smem_u32(staging) + (c0 >> 6) * L::kStagingBlock + rr * 128;
            const int cbase = (c0 & 63) >> 3;  // first 16-byte piece of this 32-column chunk inside the 64-column block
#pragma unroll
            for (int t = 0; t < 4; ++t)
              ptx::st_shared_v4(blk + (((cbase + t) ^ (rr & 7)) << 4), ptx::pack_bf16x2(v[8 * t], v[8 * t + 1]),
                                ptx::pack_bf16x2(v[8 * t + 2], v[8 * t + 3]), ptx::pack_bf16x2(v[8 * t + 4], v[8 * t + 5]),
                                ptx::pack_bf16x2(v[8 * t + 6], v[8 * t + 7]));
          } else if (valid && splits > 1) {  // split-K partial product (fp32 output, zeroed by the host)
            float* dst = reinterpret_cast<float*>(p.out) + static_cast<long long>(row) * p.ldo + n_blk * BN + c0;
#pragma unroll
            for (int j = 0; j < 32; ++j) atomicAdd(dst + j, v[j]);
          } else if (valid && TF32 && p.split3 && p.round_tf32) {  // fp32x3 tier: the next layer's operand as hi / lo TF32 halves
            store_row_chunk_split(reinterpret_cast<float*>(p.out), static_cast<long long>(row) * p.ldo + n_blk * BN + c0, p.out_lo_off, v);
          } else if (valid) {
            store_row_chunk<TF32>(p.out, static_cast<long long>(row) * p.ldo + n_blk * BN + c0, v, p.out_f32 != 0,
                                  p.round_tf32 != 0);
          }
        }
        ptx::tc_fence_before();
        if (STAGED) ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA store
        __syncwarp();
        LRN_STAMP(stamp, p.dbg, it * 8 + 5);  // accumulator drained
        if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bar_tempty[as]), 0));
        if (STAGED) {
          ptx::named_bar_sync(2 + half, 128);
          if (issuer) {
#pragma unroll
            for (int b = 0; b < kHalfCols / 64; ++b) {
              const int blk = half * (kHalfCols / 64) + b;
              ptx::tma_store_2d(&tmOut, staging + blk * L::kStagingBlock, p.out_col0 + n_blk * BN + blk * 64,
                                m_blk * 2 * BM + static_cast<int>(rank) * BM);
            }
            ptx::bulk_commit();
          }
        }
      } else {
        const int rf = it & 1;  // region of F_t; G_t is in the other one
        const long long grow = p.row0 + row;
        const long long seg = valid ? grow / p.npts : 0;
        const int n_in_seg = valid ? static_cast<int>(grow - seg * p.npts) : 0;
        const long long seg_lo = __shfl_sync(0xffffffffu, seg, 0);
        const bool uniform = !GENERAL || __all_sync(0xffffffffu, valid && seg == seg_lo);
        long long seg_hi = seg_lo;
        if (GENERAL && !uniform) {
          const unsigned vm = __ballot_sync(0xffffffffu, valid);
          seg_hi = vm ? __shfl_sync(0xffffffffu, seg, 31 - __clz(vm)) : seg_lo - 1;
        }
        const bool stamp = p.dbg && cluster_id == 0 && leader && warp == 2 && lane == 0 && it < 16;
        if (kPdl && it == 0) ptx::grid_dependency_wait();  // pooling atomics and output stores only after the chain kernel

        // ---- phase A: G_t -> gamma = 0.5 + 0.5 * sigmoid(G + bg), kept in registers (16-bit fixed point)
        uint32_t gq[kHalfCols / 2];
        const bool exact = TF32 && p.exact_gate;  // fp32x3 tier: G stays in tensor memory until phase B (no 16-bit gamma)
        ptx::mbar_wait(&bar_tfull[rf ^ 1], it & 1);
        ptx::tc_fence_after();
        LRN_STAMP(stamp, p.dbg, it * 8 + 2);  // G ready
#pragma unroll
        for (int i = 0; i < (exact ? 0 : kChunks); ++i) {  // both phases hide under the next main loop: no need to pipeline the loads
          const int c0 = col_lo + 32 * i;
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(t_lane + (rf ^ 1) * BN + c0, r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float z0 = __uint_as_float(r[j]) + sb[BN + c0 + j];
            const float z1 = __uint_as_float(r[j + 1]) + sb[BN + c0 + j + 1];
            gq[16 * i + j / 2] = gamma_pack(0.5f + __fdividef(0.5f, 1.f + __expf(-z0)),
                                            0.5f + __fdividef(0.5f, 1.f + __expf(-z1)));
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0 && !exact) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bar_tempty[rf ^ 1]), 0));  // G region drained
        LRN_STAMP(stamp, p.dbg, it * 8 + 3);  // phase A done

        // ---- phase B: v = relu(F_t + bf) * gamma, stores, pooling
        ptx::mbar_wait(&bar_tfull[rf], it & 1);
        ptx::tc_fence_after();
        LRN_STAMP(stamp, p.dbg, it * 8 + 4);  // F ready
        {
#pragma unroll
          for (int i = 0; i < kChunks; ++i) {
            const int c0 = col_lo + 32 * i;
            uint32_t r[32];
            ptx::tmem_ld_32x32b_x32(t_lane + rf * BN + c0, r);
            ptx::tmem_ld_wait();
            float v[32];
            if (exact) {  // gate in full fp32: 0.5 + 0.5 / (1 + exp(-z)), src/model.py:54-55
              uint32_t rg[32];
              ptx::tmem_ld_32x32b_x32(t_lane + (rf ^ 1) * BN + c0, rg);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float f = fmaxf(__uint_as_float(r[j]) + sb[c0 + j], 0.f);
                const float z = __uint_as_float(rg[j]) + sb[BN + c0 + j];
                v[j] = valid ? f * (0.5f + __fdiv_rn(0.5f, 1.f + expf(-z))) : 0.f;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                const float f0 = fmaxf(__uint_as_float(r[j]) + sb[c0 + j], 0.f);
                const float f1 = fmaxf(__uint_as_float(r[j + 1]) + sb[c0 + j + 1], 0.f);
                const uint32_t g = gq[16 * i + j / 2];
                v[j] = valid ? f0 * gamma_lo(g) : 0.f;
                v[j + 1] = valid ? f1 * gamma_hi(g) : 0.f;
              }
            }
            const int ch0 = n_blk * BN + c0;
            if ((p.flags & FUSE_STORE_CN) && valid) {
              float* dst = p.fused_cn + (seg * 1024 + ch0) * p.npts + n_in_seg;
#pragma unroll
              for (int j = 0; j < 32; ++j) dst[static_cast<long long>(j) * p.npts] = v[j];
            }
            if ((p.flags & FUSE_STORE_PM) && valid) {
              if (TF32 && p.split3)
                store_row_chunk_split(reinterpret_cast<float*>(p.fused_pm), static_cast<long long>(row) * 2048 + ch0, 1024, v);
              else
                store_row_chunk<TF32>(p.fused_pm, static_cast<long long>(row) * 1024 + ch0, v, TF32, TF32);
            }
            if (p.flags & (FUSE_POOL | FUSE_ARGMAX)) {
              if (!GENERAL || (uniform && !(p.flags & FUSE_ARGMAX))) {
                float mx, sm;
                pool_chunk_smem(v, scratch, lane, mx, sm);
                float* gf = p.global_feat + seg_lo * 2048 + ch0 + lane;
                if (mx > 0.f) atomicMax(reinterpret_cast<int*>(gf), __float_as_int(mx));
                if (sm > 0.f) atomicAdd(gf + 1024, sm * p.inv_npts);
              } else if (uniform) {
                pool_chunk(v, true, seg_lo, n_in_seg, ch0, lane, p);
              } else {
                for (long long s = seg_lo; s <= seg_hi; ++s)
                  pool_chunk(v, valid && seg == s, s, n_in_seg, ch0, lane, p);
              }
            }
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        LRN_STAMP(stamp, p.dbg, it * 8 + 5);  // phase B done
        if (lane == 0) {
          ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bar_tempty[rf]), 0));  // F region drained
          if (exact) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bar_tempty[rf ^ 1]), 0));  // ... and G with it
        }
      }
    }
  }

  if (STAGED && warp >= 2 && ((warp - 2) & 3) == 0 && lane == 0) ptx::bulk_wait_all();
  // Both CTAs stay resident until every MMA that reads the peer's shared memory / signals its
  // barriers has retired (the epilogue above waited for the last commit), then free TMEM.
  ptx::tc_fence_before();
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair<kTmemCols>(tmem_base);
  }
}

}  // namespace lrn
