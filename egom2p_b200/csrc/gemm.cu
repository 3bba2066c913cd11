// bf16 GEMM on the 5th-gen tensor cores: CTA pairs (cluster 2x1x1) issuing tcgen05.mma.cta_group::2 -- a 256 x BN x 16
// MMA over the two SMs, each CTA staging its own 128 rows of A and half of the B panel -- with fp32 accumulators in each
// CTA's TMEM, operands staged by TMA (128B swizzle) through an mbarrier ring, persistent over (tile pair, k-split) work
// items with a double-buffered accumulator so the epilogue of item i overlaps the main loop of item i+1. The leader CTA
// (rank 0) issues the MMAs and owns the full / accumulator-free barriers (both producers and both CTAs' epilogue warps
// arrive on them, the peer through shared::cluster addresses); its commits are multicast to both CTAs.
//
// Warp roles per CTA (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (leader) + TMEM owner, warps 2..9 = epilogue
// (two warps per TMEM lane quarter, each owning half of the tile's columns): TMEM -> registers -> (+bias, +residual,
// or the cross-entropy transforms) -> swizzled smem box -> TMA store. Split-K work items (wgrad: few output tiles,
// very long K) accumulate with TMA reduce-add, so there are no per-thread atomics and no bounds code.
//
// Operand majors (see include/egom2p_b200.h): K-major tiles are [rows][64 k] (one TMA box); MN-major tiles are
// [64 k][64 mn] boxes, one per 64 rows of the tile, consumed through MN-major UMMA descriptors -- this is what lets
// dgrad (B = W stored [N][K]) and wgrad (A = dY^T, B = X^T) run without any transposed copies.
#include "common.cuh"

namespace egom2p {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;

// EPI_STORE_BIAS_BF16: EPI_STORE with bf16 output and a bias -- its own instantiation, so that the bias code does not cost
// the plain stores registers.
enum { EPI_STORE = 0, EPI_CE_PARTIAL = 1, EPI_CE_DLOGITS = 2, EPI_SWIGLU_FWD = 3, EPI_SWIGLU_BWD = 4, EPI_GELU_FWD = 5,
       EPI_GELU_BWD = 6, EPI_STORE_BIAS_BF16 = 7 };

struct GemmParams {
  int M, N, K;
  int splits;  // k-splits per output tile (1 = plain store, > 1 = TMA reduce-add into c_f32)
  // EPI_STORE
  const float* bias;
  const float* addend;
  int64_t ld_add;
  int out_bf16, out_f32;
  // CE epilogues
  const int64_t* target;
  const float* lse;
  const float* gscale;
  // SwiGLU epilogues: ab = [a | b] interleaved in groups of 32 columns (bf16), row pitch ld_ab.
  // GELU backward: ab = the saved pre-activation u (bf16), row pitch ld_ab; GELU forward: ld_ab = row pitch of GELU(u).
  const uint16_t* ab;
  int64_t ld_ab;
  int v0;
  float* part_max;
  float* part_sum;
  float* tgt_logit;
};

// The kernel runs as CTA pairs (cluster 2x1x1) issuing tcgen05.mma.cta_group::2 -- a 256 x BN tile per pair, each CTA
// staging its own 128 rows of A and HALF of the B panel. A single-CTA 128 x 256 tile moves 12 KB of operands through shared
// memory per 128-cycle MMA while TMA refills the same 12 KB: ~188 B/clk against the 128 B/clk an SM's shared memory delivers,
// i.e. the tensor pipe idles a third of the time (ncu: 66 % active). The pair halves the B traffic per SM and deepens the ring.
template <int BN>
struct GemmSmem {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (BN / 2) * BK * 2;  // this CTA's half of the B panel
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BN == 256 ? 6 : 8;
  static constexpr int kStagingBytes = kEpiWarps * 4096;  // one 32-row x 128-byte swizzled box per epilogue warp (a second
                                                          // box costs a pipeline stage: measured 9 % slower, tools/bench_gemm_cold.py)
  static constexpr int kSched = 4;                         // cluster-launch-control response ring (work items in flight)
  static constexpr int kBarBytes = kSched * 16 + (2 * kStages + 4 + 2 * kSched) * 8 + 16;
  static constexpr int kTotal = kStages * kStageBytes + kStagingBytes + kBarBytes + 1024;  // + alignment slack
};

// logistic function with ONE MUFU op (tanh.approx, max relative error ~2^-11 -- below the bf16 rounding of every value it
// feeds) instead of ex2 + rcp: the SwiGLU epilogues evaluate it for every accumulator element
__device__ __forceinline__ float sigmoid_fast(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  return fmaf(0.5f, t, 0.5f);
}
// GELU of nn.GELU() (exact erf form) and its derivative Phi(u) + u * phi(u). erff is within 2 ulp of erf in fp32 and __expf
// within 2 ulp + 2^-21 relative for |arg| <= 32 (|u| <= 8): both errors are below 2^-18 relative to the results, far below
// the 2^-9 relative rounding of the bf16 values they are stored as.
__device__ __forceinline__ float gelu_erf(float u) { return 0.5f * u * (1.f + erff(u * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_erf_grad(float u) {
  return 0.5f * (1.f + erff(u * 0.70710678118654752f)) + u * 0.39894228040143268f * __expf(-0.5f * u * u);
}
__device__ __forceinline__ uint32_t box_off(int row, int chunk) {  // 16-byte chunk inside a [32][128 B] SW128 box
  return (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
}

template <int BN, bool A_MN, bool B_MN, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmCb, const __grid_constant__ CUtensorMap tmCf, const GemmParams p) {
  using S = GemmSmem<BN>;
  constexpr int kStages = S::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * S::kABytes;
  uint8_t* staging = smem + kStages * S::kStageBytes;
  constexpr int kSched = S::kSched;
  uint4* clc_resp = reinterpret_cast<uint4*>(smem + kStages * S::kStageBytes + S::kStagingBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(clc_resp + kSched);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* clc_full = tempty_bar + 2;     // response of the next work item landed (in every CTA of the pair)
  uint64_t* clc_empty = clc_full + kSched; // leader's: every reader of both CTAs is done with the slot
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(clc_empty + kSched);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (p.M + BM - 1) / BM, n_tiles = (p.N + BN - 1) / BN;
  const int k_blocks = (p.K + BK - 1) / BK;
  const int splits = p.splits;
  const int kb_per = (k_blocks + splits - 1) / splits;
  // Pair mode: the two CTAs of a pair walk the same work items; rank r owns M tile 2 * pair + r (its 128 rows of A and of
  // the accumulator) and stages the rows [n0 + r * BN/2, +BN/2) of B. A pair past the last M tile still takes part in the
  // loads; its TMA reads are zero-filled and its stores are clipped.
  // Work distribution: the grid holds one pair per work item; a pair starts on its own item and then keeps taking over the
  // items of pairs that have not been launched yet (cluster launch control), so the kernel is persistent -- accumulators
  // double-buffered across items -- without a static item -> SM assignment. With a static assignment one SM held by another
  // resident kernel (NCCL's all-reduce under DDP) makes the displaced pair run its whole share after everybody else:
  // 1.6x on the qkv projection (tools/bench_gemm_corun.py).
  constexpr int cl = 2;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  // One request per processed item, issued by the leader's producer warp when it starts the item; every role of both CTAs
  // reads the response after its own work on the item. Returns false when nothing was left to take over.
  auto next_item = [&](int it, int& item, bool is_scheduler) -> bool {
    const int slot = it % kSched;
    mbar_wait(&clc_full[slot], (it / kSched) & 1);
    int x;
    const bool valid = clc_decode(&clc_resp[slot], x);
    fence_async_smem();   // the generic-proxy read is ordered before the async-proxy write of the slot's next response
    __syncwarp();
    if (lane == 0 && !is_scheduler) {
      if (leader) mbar_arrive(&clc_empty[slot]);
      else mbar_arrive_cluster(cluster_map(&clc_empty[slot], 0));
    }
    item = x / cl;
    return valid;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], cl);   // pair: both producers arrive (with their byte counts) on the LEADER's barrier
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], cl * kEpiWarps);  // pair: the epilogue warps of both CTAs release the leader's barrier
    }
    for (int i = 0; i < kSched; ++i) {
      mbar_init(&clc_full[i], 1);
      mbar_init(&clc_empty[i], cl * kEpiWarps + 2);  // + the leader's MMA warp + the peer's producer warp
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_pair<2 * BN>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync();  // the peer's mbarriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // The whole warp walks the loop (addresses / coordinates stay in uniform registers); one elected lane issues.
    int stage = 0;
    uint32_t phase = 0;
    int item = blockIdx.x / cl;
    for (int it = 0;; ++it) {
      if (leader) {  // ask for the item after this one now: the answer is there long before this item's k loop ends
        const int slot = it % kSched;
        if (elect_one()) {
          mbar_wait(&clc_empty[slot], ((it / kSched) & 1) ^ 1);
          mbar_expect_tx(&clc_full[slot], 16);
          mbar_expect_tx_cluster(cluster_map(&clc_full[slot], 1), 16);
          clc_try_cancel_multicast(&clc_resp[slot], &clc_full[slot]);
        }
        __syncwarp();
      }
      const int tile = item / splits, split = item - tile * splits;
      const int m0 = ((tile / n_tiles) * cl + (int)crank) * BM, n0 = (tile % n_tiles) * BN;
      const int kb0 = split * kb_per, kb1 = min(k_blocks, kb0 + kb_per);
      for (int kb = kb0; kb < kb1; ++kb) {
        const int k0 = kb * BK;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* a = sA + stage * S::kABytes;
        uint8_t* b = sB + stage * S::kBBytes;
        if (elect_one()) {  // bytes and completions are credited to the leader's barrier (the one its MMA warp waits on)
          if (leader) mbar_expect_tx(&full_bar[stage], S::kStageBytes);
          else mbar_expect_tx_cluster(cluster_map(&full_bar[stage], 0), S::kStageBytes);
          if (!A_MN) {
            tma_load_2d_pair(a, &tmA, &full_bar[stage], k0, m0);
          } else {
#pragma unroll
            for (int h = 0; h < BM / 64; ++h) tma_load_2d_pair(a + h * 8192, &tmA, &full_bar[stage], m0 + h * 64, k0);
          }
          if (!B_MN) {
            tma_load_2d_pair(b, &tmB, &full_bar[stage], k0, n0 + (int)crank * (BN / 2));
          } else {
#pragma unroll
            for (int h = 0; h < BN / 128; ++h)
              tma_load_2d_pair(b + h * 8192, &tmB, &full_bar[stage], n0 + ((int)crank * (BN / 128) + h) * 64, k0);
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (!next_item(it, item, leader)) break;
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // Warp-uniform loop; descriptors are built once per stage in uniform registers and advanced by a constant per
    // k-step, so each tcgen05.mma costs a couple of instructions to issue (the tensor pipe needs one every 128 cycles).
    constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);  // M = 256 over the pair
    constexpr uint64_t kStepA = A_MN ? (2048 >> 4) : (32 >> 4), kStepB = B_MN ? (2048 >> 4) : (32 >> 4);
    int stage = 0;
    uint32_t phase = 0;
    int item = blockIdx.x / cl;
    for (int it = 0; leader; ++it) {  // pair: only the leader CTA issues
      const int split = item % splits;
      const int kb0 = split * kb_per, kb1 = min(k_blocks, kb0 + kb_per);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(sA + stage * S::kABytes);
        const uint32_t b_addr = smem_u32(sB + stage * S::kBBytes);
        const uint64_t da0 = A_MN ? umma_desc_mnmajor_sw128(a_addr, 8192) : umma_desc_kmajor_sw128(a_addr);
        const uint64_t db0 = B_MN ? umma_desc_mnmajor_sw128(b_addr, 8192) : umma_desc_kmajor_sw128(b_addr);
        if (elect_one()) {
          umma_bf16_ss_pair(d_tmem, da0, db0, idesc, kb > kb0 ? 1u : 0u);
#pragma unroll
          for (int k = 1; k < BK / 16; ++k) umma_bf16_ss_pair(d_tmem, da0 + k * kStepA, db0 + k * kStepB, idesc, 1u);
          umma_commit_pair(&empty_bar[stage]);                    // frees the stage in both CTAs
          if (kb == kb1 - 1) umma_commit_pair(&tfull_bar[acc]);   // accumulator halves ready in both CTAs
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (!next_item(it, item, false)) break;
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    const int q = warp & 3;              // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;    // which half of the tile's columns
    uint8_t* box = staging + (warp - 2) * 4096;
    constexpr int kHalfCols = BN / 2;
    int item = blockIdx.x / cl;
    for (int it = 0;; ++it) {
      const int tile = item / splits;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n_blk = tile % n_tiles;
      const int m0 = ((tile / n_tiles) * cl + (int)crank) * BM, n0 = n_blk * BN + half * kHalfCols;
      const int row0 = m0 + q * 32;
      const int my_row = row0 + lane;
      const bool row_ok = my_row < p.M;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + half * kHalfCols;
      float row_lse = 0.f, gs = 0.f;
      int row_tgt = -1;
      float run_max = -INFINITY, run_sum = 0.f, tl = 0.f;
      bool has_tl = false;
      if ((EPI == EPI_CE_PARTIAL || EPI == EPI_CE_DLOGITS) && row_ok) {
        row_tgt = (int)p.target[my_row] - p.v0;
        if (EPI == EPI_CE_DLOGITS) {
          row_lse = p.lse[my_row];
          gs = *p.gscale;
        }
      }
      if (EPI == EPI_CE_PARTIAL) {
#pragma unroll 1
        for (int c = 0; c < kHalfCols / 32; ++c) {
          uint32_t v[32];
          tmem_ld32(t_addr + c * 32, v);
          tmem_ld_wait();
          const int cbase = n0 + c * 32;
          float cm = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float f = (cbase + j < p.N) ? __uint_as_float(v[j]) : -INFINITY;
            cm = fmaxf(cm, f);
            if (cbase + j == row_tgt) { tl = f; has_tl = true; }
          }
          if (cm > -INFINITY) {
            const float nm = fmaxf(run_max, cm);
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (cbase + j < p.N) s += __expf(__uint_as_float(v[j]) - nm);
            run_sum = run_sum * __expf(run_max - nm) + s;
            run_max = nm;
          }
        }
        if (row_ok) {
          const int64_t o = (int64_t)(n_blk * 2 + half) * p.M + my_row;
          p.part_max[o] = run_max;
          p.part_sum[o] = run_sum;
          if (has_tl) p.tgt_logit[my_row] = tl;
        }
      } else if (EPI == EPI_SWIGLU_FWD) {
        // ---- fc1|fc3 GEMM: accumulator columns come in groups of 64 = 32 x a | 32 x b (interleaved weight rows).
        // Per 128 columns: store the two pre-activation boxes (bf16, saved for backward) and one box of
        // g = silu(a) * b (64 columns) -- the operand of the fc2 GEMM (egom2p_utils.py:167-169).
#pragma unroll 1
        for (int c = 0; c < kHalfCols / 128; ++c) {
          uint32_t gp[32];  // 64 packed bf16 gate values
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            uint32_t v0[32], v1[32];
            tmem_ld32(t_addr + c * 128 + hh * 64, v0);
            tmem_ld32(t_addr + c * 128 + hh * 64 + 32, v1);
            tmem_ld_wait();
            const int cbase = n0 + c * 128 + hh * 64;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float a0 = __uint_as_float(v0[2 * j]), a1 = __uint_as_float(v0[2 * j + 1]);
              const float g0 = a0 * sigmoid_fast(a0) * __uint_as_float(v1[2 * j]);
              const float g1 = a1 * sigmoid_fast(a1) * __uint_as_float(v1[2 * j + 1]);
              gp[hh * 16 + j] = pack_bf16(g0, g1);
            }
            tma_store_wait_read();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 pk;
              pk.x = pack_bf16(__uint_as_float(v0[8 * j + 0]), __uint_as_float(v0[8 * j + 1]));
              pk.y = pack_bf16(__uint_as_float(v0[8 * j + 2]), __uint_as_float(v0[8 * j + 3]));
              pk.z = pack_bf16(__uint_as_float(v0[8 * j + 4]), __uint_as_float(v0[8 * j + 5]));
              pk.w = pack_bf16(__uint_as_float(v0[8 * j + 6]), __uint_as_float(v0[8 * j + 7]));
              *reinterpret_cast<uint4*>(box + box_off(lane, j)) = pk;
              pk.x = pack_bf16(__uint_as_float(v1[8 * j + 0]), __uint_as_float(v1[8 * j + 1]));
              pk.y = pack_bf16(__uint_as_float(v1[8 * j + 2]), __uint_as_float(v1[8 * j + 3]));
              pk.z = pack_bf16(__uint_as_float(v1[8 * j + 4]), __uint_as_float(v1[8 * j + 5]));
              pk.w = pack_bf16(__uint_as_float(v1[8 * j + 6]), __uint_as_float(v1[8 * j + 7]));
              *reinterpret_cast<uint4*>(box + box_off(lane, j + 4)) = pk;
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0 && row0 < p.M && cbase < p.N) {
              tma_store_2d(&tmCb, box, cbase, row0);
              tma_store_commit();
            }
          }
          tma_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(box + box_off(lane, j)) = make_uint4(gp[4 * j], gp[4 * j + 1], gp[4 * j + 2], gp[4 * j + 3]);
          fence_async_smem();
          __syncwarp();
          const int gbase = (n0 + c * 128) >> 1;
          if (lane == 0 && row0 < p.M && gbase < (p.N >> 1)) {
            tma_store_2d(&tmCf, box, gbase, row0);   // aux map = g (rows, N/2) bf16
            tma_store_commit();
          }
        }
      } else if (EPI == EPI_SWIGLU_BWD) {
        // ---- fc2 dgrad: acc = dg (32 columns per step); with the saved [a | b] group of the same 32 hidden units emit
        // [da | db] (64 bf16 columns, same interleaved layout): da = dg * b * silu'(a), db = dg * silu(a).
        // The saved [a | b] rows of the NEXT 32 hidden units are fetched while the current 32 are evaluated, and they are
        // fetched COALESCED (8 lanes per 128-byte row, 4 rows per instruction) and transposed through the warp's staging box:
        // one 16-byte load per lane and row otherwise costs 32 cache lines per instruction and the LSU, not the tensor pipe,
        // bounds the kernel (178 us against 93 us for the same GEMM with a plain epilogue).
        constexpr int kSteps = kHalfCols / 32;
        uint4 abuf[2][8];
        auto fetch = [&](int c, uint4 (&dst)[8]) {
          const int cbase = n0 + c * 32;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = row0 + 4 * i + (lane >> 3);
            dst[i] = (r < p.M && cbase < p.N)
                         ? __ldg(reinterpret_cast<const uint4*>(p.ab + (int64_t)r * p.ld_ab + 2 * cbase) + (lane & 7))
                         : make_uint4(0u, 0u, 0u, 0u);
          }
        };
        fetch(0, abuf[0]);
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
          uint32_t v[32];
          tmem_ld32(t_addr + c * 32, v);
          if (c + 1 < kSteps) fetch(c + 1, abuf[(c + 1) & 1]);
          const int cbase = n0 + c * 32;           // hidden-unit base of this step
          uint4 ab[8];
          tma_store_wait_read();   // the previous store out of this warp's box has been read
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) *reinterpret_cast<uint4*>(box + box_off(4 * i + (lane >> 3), lane & 7)) = abuf[c & 1][i];
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) ab[j] = *reinterpret_cast<const uint4*>(box + box_off(lane, j));  // this lane's row
          __syncwarp();            // every lane holds its row before the box is reused for the outputs
          tmem_ld_wait();
          uint32_t da[16], db[16];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 ra = ab[j], rb = ab[j + 4];
            const uint32_t aw[4] = {ra.x, ra.y, ra.z, ra.w}, bw[4] = {rb.x, rb.y, rb.z, rb.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&aw[u]));
              const float2 fb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&bw[u]));
              const float d0 = __uint_as_float(v[8 * j + 2 * u]), d1 = __uint_as_float(v[8 * j + 2 * u + 1]);
              const float s0 = sigmoid_fast(fa.x), s1 = sigmoid_fast(fa.y);
              da[4 * j + u] = pack_bf16(d0 * fb.x * (s0 * (1.f + fa.x * (1.f - s0))), d1 * fb.y * (s1 * (1.f + fa.y * (1.f - s1))));
              db[4 * j + u] = pack_bf16(d0 * fa.x * s0, d1 * fa.y * s1);
            }
          }
          uint8_t* bx = box;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            *reinterpret_cast<uint4*>(bx + box_off(lane, j)) = make_uint4(da[4 * j], da[4 * j + 1], da[4 * j + 2], da[4 * j + 3]);
            *reinterpret_cast<uint4*>(bx + box_off(lane, j + 4)) = make_uint4(db[4 * j], db[4 * j + 1], db[4 * j + 2], db[4 * j + 3]);
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {   // (an empty group when the box is out of range keeps the wait_group accounting uniform)
            if (row0 < p.M && cbase < p.N) tma_store_2d(&tmCb, bx, 2 * cbase, row0);   // output map = dab (rows, 2N) bf16
            tma_store_commit();
          }
        }
      } else if constexpr (EPI == EPI_GELU_FWD) {
        // ---- fc1 GEMM: u = acc + b1 and GELU(u), 64 columns (one 128-byte box row) per step. The u box (bf16, saved for
        // backward) and the GELU(u) box (bf16, the operand of the fc2 GEMM) leave through the warp's staging box in turn.
        auto store_box = [&](const uint32_t (&a)[32], const uint32_t (&b)[32], const CUtensorMap* map, int cbase) {
          tma_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            *reinterpret_cast<uint4*>(box + box_off(lane, j)) =
                make_uint4(pack_bf16(__uint_as_float(a[8 * j + 0]), __uint_as_float(a[8 * j + 1])),
                           pack_bf16(__uint_as_float(a[8 * j + 2]), __uint_as_float(a[8 * j + 3])),
                           pack_bf16(__uint_as_float(a[8 * j + 4]), __uint_as_float(a[8 * j + 5])),
                           pack_bf16(__uint_as_float(a[8 * j + 6]), __uint_as_float(a[8 * j + 7])));
            *reinterpret_cast<uint4*>(box + box_off(lane, j + 4)) =
                make_uint4(pack_bf16(__uint_as_float(b[8 * j + 0]), __uint_as_float(b[8 * j + 1])),
                           pack_bf16(__uint_as_float(b[8 * j + 2]), __uint_as_float(b[8 * j + 3])),
                           pack_bf16(__uint_as_float(b[8 * j + 4]), __uint_as_float(b[8 * j + 5])),
                           pack_bf16(__uint_as_float(b[8 * j + 6]), __uint_as_float(b[8 * j + 7])));
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (row0 < p.M && cbase < p.N) tma_store_2d(map, box, cbase, row0);
            tma_store_commit();
          }
        };
#pragma unroll 1
        for (int c = 0; c < kHalfCols / 64; ++c) {
          uint32_t v0[32], v1[32];
          tmem_ld32(t_addr + c * 64, v0);
          tmem_ld32(t_addr + c * 64 + 32, v1);
          tmem_ld_wait();
          const int cbase = n0 + c * 64;
          if (p.bias) {   // N % 64 == 0: the 64 columns are all inside or all outside
            if (cbase < p.N) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 ba = __ldg(reinterpret_cast<const float4*>(p.bias + cbase) + j);
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + cbase + 32) + j);
                v0[4 * j + 0] = __float_as_uint(__uint_as_float(v0[4 * j + 0]) + ba.x);
                v0[4 * j + 1] = __float_as_uint(__uint_as_float(v0[4 * j + 1]) + ba.y);
                v0[4 * j + 2] = __float_as_uint(__uint_as_float(v0[4 * j + 2]) + ba.z);
                v0[4 * j + 3] = __float_as_uint(__uint_as_float(v0[4 * j + 3]) + ba.w);
                v1[4 * j + 0] = __float_as_uint(__uint_as_float(v1[4 * j + 0]) + bb.x);
                v1[4 * j + 1] = __float_as_uint(__uint_as_float(v1[4 * j + 1]) + bb.y);
                v1[4 * j + 2] = __float_as_uint(__uint_as_float(v1[4 * j + 2]) + bb.z);
                v1[4 * j + 3] = __float_as_uint(__uint_as_float(v1[4 * j + 3]) + bb.w);
              }
            }
          }
          store_box(v0, v1, &tmCb, cbase);   // u
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            v0[j] = __float_as_uint(gelu_erf(__uint_as_float(v0[j])));
            v1[j] = __float_as_uint(gelu_erf(__uint_as_float(v1[j])));
          }
          store_box(v0, v1, &tmCf, cbase);   // aux map = GELU(u) (rows, N) bf16
        }
      } else if constexpr (EPI == EPI_GELU_BWD) {
        // ---- fc2 dgrad: acc = dh, 64 columns per step; with the saved pre-activation u of the same columns emit
        // du = dh * GELU'(u) (bf16). u is fetched coalesced (8 lanes per 128-byte row, 4 rows per instruction) and
        // transposed through the warp's staging box, as in the SwiGLU backward; its loads are in flight while the
        // accumulator is read. (A one-step-ahead prefetch, as there, spills at the 168-register cap.)
        constexpr int kSteps = kHalfCols / 64;
        uint4 ubuf[8];
        auto fetch = [&](int c, uint4 (&dst)[8]) {
          const int cbase = n0 + c * 64;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = row0 + 4 * i + (lane >> 3);
            dst[i] = (r < p.M && cbase < p.N)
                         ? __ldg(reinterpret_cast<const uint4*>(p.ab + (int64_t)r * p.ld_ab + cbase) + (lane & 7))
                         : make_uint4(0u, 0u, 0u, 0u);
          }
        };
#pragma unroll 1
        for (int c = 0; c < kSteps; ++c) {
          uint32_t v[32];
          fetch(c, ubuf);
          tmem_ld32(t_addr + c * 64, v);
          const int cbase = n0 + c * 64;
          uint4 ur[8];
          tma_store_wait_read();   // the previous store out of this warp's box has been read
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) *reinterpret_cast<uint4*>(box + box_off(4 * i + (lane >> 3), lane & 7)) = ubuf[i];
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) ur[j] = *reinterpret_cast<const uint4*>(box + box_off(lane, j));  // this lane's row
          __syncwarp();            // every lane holds its row before the box is reused for the output
          // the 64 accumulator columns are read in two halves of 32: one half in registers at a time (no spills)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            if (hh) tmem_ld32(t_addr + c * 64 + 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 4 * hh; j < 4 * hh + 4; ++j) {
              const uint32_t uw[4] = {ur[j].x, ur[j].y, ur[j].z, ur[j].w};
              uint32_t o[4];
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 fu = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&uw[t]));
                const int k = 8 * (j - 4 * hh) + 2 * t;
                o[t] = pack_bf16(__uint_as_float(v[k]) * gelu_erf_grad(fu.x), __uint_as_float(v[k + 1]) * gelu_erf_grad(fu.y));
              }
              *reinterpret_cast<uint4*>(box + box_off(lane, j)) = make_uint4(o[0], o[1], o[2], o[3]);
            }
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {   // (an empty group when the box is out of range keeps the wait_group accounting uniform)
            if (row0 < p.M && cbase < p.N) tma_store_2d(&tmCb, box, cbase, row0);   // output map = du (rows, N) bf16
            tma_store_commit();
          }
        }
      } else if (EPI == EPI_CE_DLOGITS || EPI == EPI_STORE_BIAS_BF16 || p.out_bf16) {
        // ---- bf16 output: 64 columns (one 128-byte box row) per step
#pragma unroll 1
        for (int c = 0; c < kHalfCols / 64; ++c) {
          uint32_t v0[32], v1[32];
          tmem_ld32(t_addr + c * 64, v0);
          tmem_ld32(t_addr + c * 64 + 32, v1);
          tmem_ld_wait();
          const int cbase = n0 + c * 64;
          if (EPI == EPI_CE_DLOGITS) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float p0 = __expf(__uint_as_float(v0[j]) - row_lse), p1 = __expf(__uint_as_float(v1[j]) - row_lse);
              if (cbase + j == row_tgt) p0 -= 1.f;
              if (cbase + 32 + j == row_tgt) p1 -= 1.f;
              v0[j] = __float_as_uint(p0 * gs);
              v1[j] = __float_as_uint(p1 * gs);
            }
          }
          if constexpr (EPI == EPI_STORE_BIAS_BF16) {   // N % 8 == 0: a float4 of the bias is either wholly inside or wholly outside
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int k = (j & 7) * 4, col = cbase + (j >> 3) * 32 + k;
              if (col < p.N) {
                const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + col));
                uint32_t* v = j < 8 ? v0 : v1;
                v[k + 0] = __float_as_uint(__uint_as_float(v[k + 0]) + bv.x);
                v[k + 1] = __float_as_uint(__uint_as_float(v[k + 1]) + bv.y);
                v[k + 2] = __float_as_uint(__uint_as_float(v[k + 2]) + bv.z);
                v[k + 3] = __float_as_uint(__uint_as_float(v[k + 3]) + bv.w);
              }
            }
          }
          uint8_t* bx = box;
          tma_store_wait_read();   // previous store out of this warp's box has been read
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 pk;
            pk.x = pack_bf16(__uint_as_float(v0[8 * j + 0]), __uint_as_float(v0[8 * j + 1]));
            pk.y = pack_bf16(__uint_as_float(v0[8 * j + 2]), __uint_as_float(v0[8 * j + 3]));
            pk.z = pack_bf16(__uint_as_float(v0[8 * j + 4]), __uint_as_float(v0[8 * j + 5]));
            pk.w = pack_bf16(__uint_as_float(v0[8 * j + 6]), __uint_as_float(v0[8 * j + 7]));
            *reinterpret_cast<uint4*>(bx + box_off(lane, j)) = pk;
            pk.x = pack_bf16(__uint_as_float(v1[8 * j + 0]), __uint_as_float(v1[8 * j + 1]));
            pk.y = pack_bf16(__uint_as_float(v1[8 * j + 2]), __uint_as_float(v1[8 * j + 3]));
            pk.z = pack_bf16(__uint_as_float(v1[8 * j + 4]), __uint_as_float(v1[8 * j + 5]));
            pk.w = pack_bf16(__uint_as_float(v1[8 * j + 6]), __uint_as_float(v1[8 * j + 7]));
            *reinterpret_cast<uint4*>(bx + box_off(lane, j + 4)) = pk;
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (row0 < p.M && cbase < p.N) tma_store_2d(&tmCb, bx, cbase, row0);
            tma_store_commit();
          }
        }
      } else {
        // ---- fp32 output (+bias, +residual / accumulate): 32 columns (one 128-byte box row) per step. The residual row
        // of the NEXT step is fetched while the current one is written out: the epilogue of the fp32-residual GEMMs (proj,
        // fc2: 200 MB in + out per launch at b = 16) is bound by these global-load round trips, not by its math.
        constexpr int kSteps = kHalfCols / 32;
        const bool use_add = p.addend && splits == 1 && row_ok;
        float4 abuf[2][8];
        auto fetch = [&](int c, float4 (&dst)[8]) {
          const int cbase = n0 + c * 32;
          const float* arow = p.addend + (int64_t)my_row * p.ld_add + cbase;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            dst[j] = (use_add && cbase + 4 * j < p.N) ? __ldg(reinterpret_cast<const float4*>(arow + 4 * j)) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        if (p.addend) fetch(0, abuf[0]);
#pragma unroll
        for (int c = 0; c < kSteps; ++c) {
          uint32_t v[32];
          tmem_ld32(t_addr + c * 32, v);
          if (p.addend && c + 1 < kSteps) fetch(c + 1, abuf[(c + 1) & 1]);
          tmem_ld_wait();
          const int cbase = n0 + c * 32;
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (cbase + 4 * j < p.N) {
                const float4 bv = *reinterpret_cast<const float4*>(p.bias + cbase + 4 * j);
                v[4 * j + 0] = __float_as_uint(__uint_as_float(v[4 * j + 0]) + bv.x);
                v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + bv.y);
                v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + bv.z);
                v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + bv.w);
              }
            }
          }
          if (p.addend) {
            const float4(&av)[8] = abuf[c & 1];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              v[4 * j + 0] = __float_as_uint(__uint_as_float(v[4 * j + 0]) + av[j].x);
              v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + av[j].y);
              v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + av[j].z);
              v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + av[j].w);
            }
          }
          uint8_t* bx = box;
          tma_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(bx + box_off(lane, j)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (row0 < p.M && cbase < p.N) {
              if (splits > 1) tma_reduce_add_2d(&tmCf, bx, cbase, row0);
              else tma_store_2d(&tmCf, bx, cbase, row0);
            }
            tma_store_commit();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tempty_bar[acc]);
        else mbar_arrive_cluster(cluster_map(&tempty_bar[acc], 0));
      }
      if (!next_item(it, item, false)) break;
    }
    tma_store_wait_all();  // global writes complete before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync();  // no CTA leaves while its peer may still signal its mbarriers / read its smem
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair<2 * BN>(tmem_base);
  }
}

static int sm_count() { return device_sm_count(); }

template <int BN, bool A_MN, bool B_MN, int EPI>
static int launch_gemm(const uint16_t* A, const uint16_t* B, int64_t lda, int64_t ldb, uint16_t* c_bf16, float* c_f32,
                       int64_t ldc, GemmParams p, cudaStream_t stream) {
  using S = GemmSmem<BN>;
  CUtensorMap tmA, tmB, tmCb, tmCf;
  int rc;
  if (!A_MN) rc = make_tmap_bf16_2d(&tmA, A, p.M, p.K, lda, BM, BK);
  else       rc = make_tmap_bf16_2d(&tmA, A, p.K, p.M, lda, BK, 64);
  if (rc) return rc;
  if (!B_MN) rc = make_tmap_bf16_2d(&tmB, B, p.N, p.K, ldb, BN / 2, BK);
  else       rc = make_tmap_bf16_2d(&tmB, B, p.K, p.N, ldb, BK, 64);
  if (rc) return rc;
  tmCb = tmA;
  tmCf = tmA;
  if (EPI == EPI_GELU_BWD) {            // c_bf16 = du (M, N)
    if ((rc = make_tmap_2d(&tmCb, c_bf16, 2, p.M, p.N, ldc, 32, 64))) return rc;
  } else if (EPI == EPI_GELU_FWD) {     // c_bf16 = u (M, N); c_f32 slot carries GELU(u) (M, N) bf16 with pitch p.ld_ab
    if ((rc = make_tmap_2d(&tmCb, c_bf16, 2, p.M, p.N, ldc, 32, 64))) return rc;
    if ((rc = make_tmap_2d(&tmCf, c_f32, 2, p.M, p.N, p.ld_ab, 32, 64))) return rc;
  } else if (EPI == EPI_SWIGLU_BWD) {   // c_bf16 = dab (M, 2N)
    if ((rc = make_tmap_2d(&tmCb, c_bf16, 2, p.M, 2 * (uint64_t)p.N, ldc, 32, 64))) return rc;
  } else if (EPI == EPI_SWIGLU_FWD) {   // c_bf16 = ab (M, N); c_f32 slot carries g (M, N/2) bf16 with pitch p.ld_ab
    if ((rc = make_tmap_2d(&tmCb, c_bf16, 2, p.M, p.N, ldc, 32, 64))) return rc;
    if ((rc = make_tmap_2d(&tmCf, c_f32, 2, p.M, (uint64_t)p.N / 2, p.ld_ab, 32, 64))) return rc;
  } else {
    if (c_bf16 && (rc = make_tmap_2d(&tmCb, c_bf16, 2, p.M, p.N, ldc, 32, 64))) return rc;
    if (c_f32 && (rc = make_tmap_2d(&tmCf, c_f32, 4, p.M, p.N, ldc, 32, 32))) return rc;
  }
  p.out_bf16 = c_bf16 != nullptr;
  p.out_f32 = c_f32 != nullptr;
  auto kern = gemm_kernel<BN, A_MN, B_MN, EPI>;
  static std::atomic<uint64_t> attr_done{0};   // one flag set per template instantiation
  if ((rc = ensure_dyn_smem(kern, S::kTotal, attr_done, "gemm"))) return rc;
  const int sms = sm_count();
  const int k_blocks = (p.K + BK - 1) / BK;
  // split-K: only for fp32 accumulate/plain outputs, when the output tiles cannot fill the machine and K is long
  int splits = 1;
  // work units the persistent workers (CTA pairs) share: 256-row tile pairs
  const int units = (((p.M + BM - 1) / BM + 1) / 2) * ((p.N + BN - 1) / BN);
  const int workers = sms / 2;
  if (EPI == EPI_STORE && !c_bf16 && !p.bias && (!p.addend || p.addend == c_f32) && units < 3 * workers && k_blocks >= 16) {
    // the number of splits that fills r whole rounds of workers best (r = 1..4; ties: fewer rounds = fewer reduce-adds).
    // Also taken when the tiles alone already exceed one round but quantise badly (the head's dW chunks: 96 tiles on 74
    // pairs = 65 % of two rounds; 3 splits = 288 items = 97 % of four rounds).
    float best = (float)units / (float)(((units + workers - 1) / workers) * workers);
    if (units < workers) best = 0.f;
    for (int r = 1; r <= 4; ++r) {
      int sp = workers * r / units;
      sp = sp < k_blocks / 8 ? sp : k_blocks / 8;
      if (sp < 1) sp = 1;
      const float util = (float)(units * sp) / (float)(((units * sp + workers - 1) / workers) * workers);
      if (util > best + (units < workers ? 0.02f : 0.10f)) { best = util; splits = sp; }
    }
    const int kb_per = (k_blocks + splits - 1) / splits;
    splits = (k_blocks + kb_per - 1) / kb_per;  // no empty splits
  }
  p.splits = splits;
  if (splits > 1 && !p.addend) {  // reduce-add needs a zeroed destination (an aliased addend means "accumulate into C")
    cudaError_t e = cudaMemset2DAsync(c_f32, ldc * sizeof(float), 0, (size_t)p.N * sizeof(float), p.M, stream);
    if (e != cudaSuccess) { set_error("gemm: memset: %s", cudaGetErrorString(e)); return EGOM2P_ERR_CUDA; }
  }
  // CTA pairs: clusters of 2 along x
  const int pair_items = (((p.M + BM - 1) / BM + 1) / 2) * ((p.N + BN - 1) / BN) * splits;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(kGemmThreads); cfg.dynamicSmemBytes = S::kTotal; cfg.stream = stream; cfg.attrs = attr; cfg.numAttrs = 1;
  cfg.gridDim = dim3(2 * pair_items);   // one pair per work item; the pairs that get to run cancel and absorb the rest
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmCb, tmCf, p);
  if (e != cudaSuccess) { set_error("gemm: cluster launch: %s", cudaGetErrorString(e)); return EGOM2P_ERR_CUDA; }
  return check_launch("gemm_bf16");
}

template <int EPI>
static int dispatch_gemm(const uint16_t* A, const uint16_t* B, int64_t lda, int64_t ldb, int a_mn, int b_mn,
                         uint16_t* c_bf16, float* c_f32, int64_t ldc, const GemmParams& p, cudaStream_t stream) {
  // BN = 256 halves B re-reads per tile; BN = 128 gives better wave quantisation on small problems.
  const int sms = sm_count();
  const int64_t tiles256 = (int64_t)((p.M + BM - 1) / BM) * ((p.N + 255) / 256);
  constexpr bool kStore = EPI == EPI_STORE || EPI == EPI_STORE_BIAS_BF16;
  const bool use256 = !kStore || (p.N >= 256 && (tiles256 >= 2 * sms || !c_bf16));
#define EGO_GEMM_CASE(BN_, AM, BMJ) return launch_gemm<BN_, AM, BMJ, EPI>(A, B, lda, ldb, c_bf16, c_f32, ldc, p, stream)
  if constexpr (EPI == EPI_SWIGLU_BWD || EPI == EPI_GELU_BWD) {  // dg / dh = dY W2 (B consumed MN-major)
    EGO_GEMM_CASE(256, false, true);
  } else if constexpr (!kStore) {  // CE / SwiGLU- and GELU-forward epilogues: K-major x K-major
    EGO_GEMM_CASE(256, false, false);
  } else if constexpr (EPI == EPI_STORE_BIAS_BF16) {  // biased projections (qkv, q, kv): K-major x K-major
    if (use256) EGO_GEMM_CASE(256, false, false);
    EGO_GEMM_CASE(128, false, false);
  } else if (use256) {
    if (!a_mn && !b_mn) EGO_GEMM_CASE(256, false, false);
    if (!a_mn && b_mn) EGO_GEMM_CASE(256, false, true);
    if (a_mn && b_mn) EGO_GEMM_CASE(256, true, true);
    EGO_GEMM_CASE(256, true, false);
  } else {
    if (!a_mn && !b_mn) EGO_GEMM_CASE(128, false, false);
    if (!a_mn && b_mn) EGO_GEMM_CASE(128, false, true);
    if (a_mn && b_mn) EGO_GEMM_CASE(128, true, true);
    EGO_GEMM_CASE(128, true, false);
  }
#undef EGO_GEMM_CASE
}

}  // namespace egom2p

extern "C" int egom2p_gemm_bf16(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, int64_t lda,
                                int64_t ldb, int32_t a_mn, int32_t b_mn, const float* bias, const float* addend,
                                int64_t ld_add, uint16_t* c_bf16, float* c_f32, int64_t ldc, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(A && B && M > 0 && N > 0 && K > 0, "gemm_bf16: null operand or empty shape (M=%d N=%d K=%d)", M, N, K);
  EGO_REQUIRE((c_bf16 != nullptr) != (c_f32 != nullptr), "gemm_bf16: exactly one of c_bf16 / c_f32");
  EGO_REQUIRE(N % 4 == 0 && ldc % 4 == 0 && (!addend || ld_add % 4 == 0), "gemm_bf16: N, ldc, ld_add must be multiples of 4");
  EGO_REQUIRE(!c_bf16 || (N % 8 == 0 && ldc % 8 == 0), "gemm_bf16: bf16 output needs N, ldc multiples of 8");
  GemmParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.addend = addend; p.ld_add = ld_add;
  if (c_bf16 && bias) {
    EGO_REQUIRE(!a_mn && !b_mn && !addend, "gemm_bf16: a bias with bf16 output needs K-major A and B and no addend");
    EGO_REQUIRE(((uintptr_t)bias & 15) == 0, "gemm_bf16: bias must be 16-byte aligned");
    return dispatch_gemm<EPI_STORE_BIAS_BF16>(A, B, lda, ldb, 0, 0, c_bf16, nullptr, ldc, p, (cudaStream_t)stream);
  }
  return dispatch_gemm<EPI_STORE>(A, B, lda, ldb, a_mn, b_mn, c_bf16, c_f32, ldc, p, (cudaStream_t)stream);
}

extern "C" int egom2p_ce_partials(const uint16_t* Y, const uint16_t* W, const int64_t* target, int32_t R, int32_t V, int32_t K,
                                  int64_t ldy, int64_t ldw, float* part_max, float* part_sum, float* tgt_logit, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(Y && W && target && part_max && part_sum && tgt_logit && R > 0 && V > 0 && K > 0, "ce_partials: bad argument");
  GemmParams p{};
  p.M = R; p.N = V; p.K = K; p.target = target; p.v0 = 0; p.part_max = part_max; p.part_sum = part_sum; p.tgt_logit = tgt_logit;
  return dispatch_gemm<EPI_CE_PARTIAL>(Y, W, ldy, ldw, 0, 0, nullptr, nullptr, 0, p, (cudaStream_t)stream);
}

extern "C" int egom2p_ce_dlogits(const uint16_t* Y, const uint16_t* W, const int64_t* target, const float* lse,
                                 const float* gscale, int32_t R, int32_t v0, int32_t Vc, int32_t K, int64_t ldy, int64_t ldw,
                                 uint16_t* dlogits, int64_t ldd, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(Y && W && target && lse && gscale && dlogits && R > 0 && Vc > 0 && K > 0 && v0 >= 0, "ce_dlogits: bad argument");
  EGO_REQUIRE(Vc % 8 == 0 && ldd % 8 == 0, "ce_dlogits: Vc and ldd must be multiples of 8");
  GemmParams p{};
  p.M = R; p.N = Vc; p.K = K; p.target = target; p.lse = lse; p.gscale = gscale; p.v0 = v0;
  return dispatch_gemm<EPI_CE_DLOGITS>(Y, W + (int64_t)v0 * ldw, ldy, ldw, 0, 0, dlogits, nullptr, ldd, p, (cudaStream_t)stream);
}

extern "C" int egom2p_gemm_swiglu_fwd(const uint16_t* X, const uint16_t* W13, int32_t M, int32_t N2, int32_t K, int64_t ldx,
                                      int64_t ldw, uint16_t* ab, int64_t ld_ab, uint16_t* g, int64_t ldg, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(X && W13 && ab && g && M > 0 && N2 > 0 && K > 0, "gemm_swiglu_fwd: bad argument");
  EGO_REQUIRE(N2 % 64 == 0 && ld_ab % 8 == 0 && ldg % 8 == 0, "gemm_swiglu_fwd: 2*hidden must be a multiple of 64 (32-wide a|b groups)");
  GemmParams p{};
  p.M = M; p.N = N2; p.K = K; p.ld_ab = ldg;
  return dispatch_gemm<EPI_SWIGLU_FWD>(X, W13, ldx, ldw, 0, 0, ab, reinterpret_cast<float*>(g), ld_ab, p, (cudaStream_t)stream);
}

extern "C" int egom2p_gemm_swiglu_bwd(const uint16_t* dY, const uint16_t* W2, const uint16_t* ab, int32_t M, int32_t hidden,
                                      int32_t K, int64_t ldy, int64_t ldw, int64_t ld_ab, uint16_t* dab, int64_t ld_dab,
                                      void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(dY && W2 && ab && dab && M > 0 && hidden > 0 && K > 0, "gemm_swiglu_bwd: bad argument");
  EGO_REQUIRE(hidden % 32 == 0 && ld_ab % 8 == 0 && ld_dab % 8 == 0, "gemm_swiglu_bwd: hidden must be a multiple of 32");
  GemmParams p{};
  p.M = M; p.N = hidden; p.K = K; p.ab = ab; p.ld_ab = ld_ab;
  return dispatch_gemm<EPI_SWIGLU_BWD>(dY, W2, ldy, ldw, 0, 1, dab, nullptr, ld_dab, p, (cudaStream_t)stream);
}

extern "C" int egom2p_gemm_gelu_fwd(const uint16_t* X, const uint16_t* W1, const float* b1, int32_t M, int32_t N, int32_t K,
                                    int64_t ldx, int64_t ldw, uint16_t* u, int64_t ld_u, uint16_t* h, int64_t ldh, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(X && W1 && u && h && M > 0 && N > 0 && K > 0, "gemm_gelu_fwd: bad argument");
  EGO_REQUIRE(N % 64 == 0 && ld_u % 8 == 0 && ldh % 8 == 0, "gemm_gelu_fwd: hidden must be a multiple of 64");
  EGO_REQUIRE(!b1 || ((uintptr_t)b1 & 15) == 0, "gemm_gelu_fwd: bias must be 16-byte aligned");
  GemmParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = b1; p.ld_ab = ldh;
  return dispatch_gemm<EPI_GELU_FWD>(X, W1, ldx, ldw, 0, 0, u, reinterpret_cast<float*>(h), ld_u, p, (cudaStream_t)stream);
}

extern "C" int egom2p_gemm_gelu_bwd(const uint16_t* dY, const uint16_t* W2, const uint16_t* u, int32_t M, int32_t hidden, int32_t K,
                                    int64_t ldy, int64_t ldw, int64_t ld_u, uint16_t* du, int64_t ld_du, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(dY && W2 && u && du && M > 0 && hidden > 0 && K > 0, "gemm_gelu_bwd: bad argument");
  EGO_REQUIRE(hidden % 64 == 0 && ld_u % 8 == 0 && ld_du % 8 == 0, "gemm_gelu_bwd: hidden must be a multiple of 64");
  GemmParams p{};
  p.M = M; p.N = hidden; p.K = K; p.ab = u; p.ld_ab = ld_u;
  return dispatch_gemm<EPI_GELU_BWD>(dY, W2, ldy, ldw, 0, 1, du, nullptr, ld_du, p, (cudaStream_t)stream);
}

namespace egom2p {
__global__ void ce_finalize_kernel(const float* __restrict__ pm, const float* __restrict__ ps, const float* __restrict__ tl,
                                   int R, int n_parts, float* __restrict__ lse, float* __restrict__ loss_sum) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float contrib = 0.f;
  if (r < R) {
    float m = -INFINITY;
    for (int t = 0; t < n_parts; ++t) m = fmaxf(m, pm[(int64_t)t * R + r]);
    float s = 0.f;
    for (int t = 0; t < n_parts; ++t) {
      const float pmv = pm[(int64_t)t * R + r];
      if (pmv > -INFINITY) s += ps[(int64_t)t * R + r] * __expf(pmv - m);
    }
    const float l = m + logf(s);
    lse[r] = l;
    contrib = l - tl[r];
  }
  contrib = warp_sum(contrib);
  __shared__ float sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = contrib;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < 8 ? sh[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0 && loss_sum) atomicAdd(loss_sum, t);
  }
}
}  // namespace egom2p

extern "C" int egom2p_ce_finalize(const float* part_max, const float* part_sum, const float* tgt_logit, int32_t R,
                                  int32_t n_tiles, float* lse, float* loss_sum, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(part_max && part_sum && tgt_logit && lse && R > 0 && n_tiles > 0, "ce_finalize: bad argument");
  ce_finalize_kernel<<<(R + 255) / 256, 256, 0, (cudaStream_t)stream>>>(part_max, part_sum, tgt_logit, R, n_tiles, lse, loss_sum);
  return check_launch("ce_finalize");
}
