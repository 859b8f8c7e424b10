// sb_gemm_bf16_tn: C[M,N] (f32) (+)= A[M,K] (bf16, K-major) * B[N,K]^T (bf16, K-major) (+ bias[N])
//
// Hand-written sm_100a GEMM used for every dense contraction on the encoder path
// (GRU input projections X*W_ih^T, their dgrad/wgrad, the output projection and its grads;
//  reference: nn.GRU / LinearND in speech/models/model.py:35-39,115-133, which reach cuDNN/cuBLAS).
//
//   * persistent grid (one CTA per SM), static tile schedule, N-fastest rasterisation so the
//     A row-panel is served from L2 to the CTAs working on its N tiles
//   * warp 0   : TMA producer (cp.async.bulk.tensor, SWIZZLE_128B boxes of 64 bf16 along K)
//   * warp 1   : tcgen05.mma issuer (one elected lane), accumulators in TMEM, 2 accumulator stages
//   * warps 2-5: epilogue (tcgen05.ld 32x32b -> bias / row-remap -> st.global or red.add)
//   * smem ring of kStages {A 128x64, B BNx64} tiles, full/empty mbarriers
//
// Roofline: tensor (bf16 dense).  Algorithmic FLOPs = 2*M*N*K per launch.
#include "common.cuh"
#include <cuda.h>
#include <stdio.h>

#include "../../include/speech_b200.h"

namespace sb {

static constexpr int BM = 128;
static constexpr int BK = 64;  // 64 bf16 = 128 bytes = one SWIZZLE_128B row

struct GemmParams {
  float* C;
  const float* bias;
  long long ldc;
  int M, N, K;
  int k_blocks_total;   // ceil(K / 64)
  int split_k;          // >= 1
  int flags;            // SB_GEMM_ACCUMULATE | SB_GEMM_ROW_REMAP
  int remap_B, remap_T, valid_B;
  int m_tiles, n_tiles;
  int tma_store;        // epilogue through swizzled smem + cp.async.bulk.tensor stores
  int a_mn, b_mn;       // operand given MN-major ([K][M] / [K][N], contraction dim slowest)
};

// MN-major operand tiles: the contraction runs over the ROWS of the global matrix ([K][MN], MN
// contiguous), which is how activations [tokens][features] look to a weight-gradient GEMM.  A TMA
// box {64 MN (inner, 128 B), 64 K rows} with SWIZZLE_128B lands as one 8 KB block that is exactly
// the canonical UMMA MN-major SWIZZLE_128B layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte
// units: 8 K-rows of 128 B per swizzle atom (SBO = 1024 B between atoms), the next 64 MN at
// LBO = 8192 B (the next box).  One MMA (K = 16) spans two atoms; the next MMA starts 2048 B on.
static constexpr int MN_BOX_BYTES = 64 * 64 * 2;
static constexpr uint32_t MN_LBO = MN_BOX_BYTES, MN_SBO = 1024, MN_KADV = 2048;

SB_DEVINL uint64_t umma_desc_sw128_mnmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((MN_LBO >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((MN_SBO >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <int BN>
struct GemmCfg {
  static constexpr int kStageBytes = (BM + BN) * BK * 2;
  static constexpr int kStagesRaw = (200 * 1024) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kAccStages = 2;
  static constexpr int kTmemColsRaw = kAccStages * BN;
  static constexpr int kTmemCols = kTmemColsRaw < 32 ? 32 : kTmemColsRaw;
  static constexpr int kStageOutBytes = 4 * 2 * 4096;   // 4 epilogue warps x 2 x [32 x 32] f32
  static constexpr int kSmemBytes =
      kStages * kStageBytes + kStageOutBytes + 1024 /*align*/ + 256 /*barriers*/;
};

template <int BN>
__global__ void __launch_bounds__(192, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmap_a,
                    const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_c, const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kAcc = Cfg::kAccStages;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte aligned tile ring (SWIZZLE_128B requirement)
  uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~static_cast<uintptr_t>(1023));
  uint8_t* out_stage = tiles + kStages * Cfg::kStageBytes;   // 1024-aligned (stage bytes are)
  uint64_t* bars = reinterpret_cast<uint64_t*>(out_stage + Cfg::kStageOutBytes);
  uint64_t* full_bar = bars;                  // [kStages]
  uint64_t* empty_bar = bars + kStages;       // [kStages]
  uint64_t* tfull_bar = bars + 2 * kStages;   // [2]
  uint64_t* tempty_bar = bars + 2 * kStages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if (p.tma_store) tma_prefetch_desc(&tmap_c);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 4);  // one arrive per epilogue warp
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles_mn = p.m_tiles * p.n_tiles;
  const int total_work = tiles_mn * p.split_k;
  const int kb_per_split = (p.k_blocks_total + p.split_k - 1) / p.split_k;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        const int split = w / tiles_mn;
        const int t = w - split * tiles_mn;
        const int m_blk = t / p.n_tiles;
        const int n_blk = t - m_blk * p.n_tiles;
        const int kb0 = split * kb_per_split;
        int kb1 = kb0 + kb_per_split;
        if (kb1 > p.k_blocks_total) kb1 = p.k_blocks_total;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = tiles + stage * Cfg::kStageBytes;
          uint8_t* sb_ = sa + BM * BK * 2;
          mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
          if (p.a_mn) {
#pragma unroll
            for (int b = 0; b < BM / 64; ++b)
              tma_load_2d(sa + b * MN_BOX_BYTES, &tmap_a, &full_bar[stage], m_blk * BM + b * 64,
                          kb * BK);
          } else {
            tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BK, m_blk * BM);
          }
          if (p.b_mn) {
#pragma unroll
            for (int b = 0; b < (BN + 63) / 64; ++b)
              tma_load_2d(sb_ + b * MN_BOX_BYTES, &tmap_b, &full_bar[stage], n_blk * BN + b * 64,
                          kb * BK);
          } else {
            tma_load_2d(sb_, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = umma_idesc_bf16_f32(BM, BN) | (p.a_mn ? (1u << 15) : 0u) |
                           (p.b_mn ? (1u << 16) : 0u);
    const uint64_t a_step = p.a_mn ? (uint64_t)(MN_KADV >> 4) : 2u;
    const uint64_t b_step = p.b_mn ? (uint64_t)(MN_KADV >> 4) : 2u;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int split = w / tiles_mn;
      const int kb0 = split * kb_per_split;
      int kb1 = kb0 + kb_per_split;
      if (kb1 > p.k_blocks_total) kb1 = p.k_blocks_total;
      if (lane == 0) mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      __syncwarp();
      tc_fence_after_sync();
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int kb = kb0; kb < kb1; ++kb) {
        if (lane == 0) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          const uint32_t sa = smem_u32(tiles + stage * Cfg::kStageBytes);
          const uint32_t sb_ = sa + BM * BK * 2;
          const uint64_t da = p.a_mn ? umma_desc_sw128_mnmajor(sa) : umma_desc_sw128_kmajor(sa);
          const uint64_t db = p.b_mn ? umma_desc_sw128_mnmajor(sb_) : umma_desc_sw128_kmajor(sb_);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // K-major: advance 16 bf16 = 32 bytes along K inside the swizzle atom (+2 in the
            // >>4 field); MN-major: 16 K-rows of 128 B = 2048 bytes
            umma_bf16_ss(tmem_d, da + a_step * k, db + b_step * k, idesc,
                         (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs retire
          if (kb == kb1 - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (kb1 <= kb0 && lane == 0) {
        // empty K range (can only happen with an over-split K): nothing accumulated
        umma_commit(&tfull_bar[acc]);
      }
      if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    // ===================== epilogue warps (2..5) =====================
    const int sub = warp & 3;  // TMEM sub-partition this warp may read: lanes [32*sub, 32*sub+32)
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool vec_ok = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
    unsigned int out_slot = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int split = w / tiles_mn;
      const int t = w - split * tiles_mn;
      const int m_blk = t / p.n_tiles;
      const int n_blk = t - m_blk * p.n_tiles;
      const int kb0 = split * kb_per_split;
      const bool has_k = kb0 < p.k_blocks_total;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after_sync();
      const int m = m_blk * BM + sub * 32 + lane;
      bool row_ok = m < p.M;
      long long out_row = m;
      if (p.flags & SB_GEMM_ROW_REMAP) {
        const int b = m % p.remap_B;
        const int tt = m / p.remap_B;
        row_ok = row_ok && (b < p.valid_B);
        out_row = (long long)b * p.remap_T + tt;
      }
      float* crow = p.C + out_row * p.ldc;
      const bool add_bias = (p.bias != nullptr) && (split == 0);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(sub * 32) << 16) + acc * BN + c * 32, v);
        tmem_ld_wait();
        const int n0 = n_blk * BN + c * 32;
        if (p.tma_store) {
          // ---- coalesced path: registers -> swizzled smem tile -> one bulk tensor store ----
          const int m0 = m_blk * BM + sub * 32;
          if (has_k && n0 < p.N && m0 < p.M) {      // warp-uniform
            uint8_t* buf = out_stage + ((warp - 2) * 2 + (out_slot & 1)) * 4096;
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o;
              o.x = __uint_as_float(v[j + 0]);
              o.y = __uint_as_float(v[j + 1]);
              o.z = __uint_as_float(v[j + 2]);
              o.w = __uint_as_float(v[j + 3]);
              if (add_bias) {
                if (n0 + j + 0 < p.N) o.x += __ldg(p.bias + n0 + j + 0);
                if (n0 + j + 1 < p.N) o.y += __ldg(p.bias + n0 + j + 1);
                if (n0 + j + 2 < p.N) o.z += __ldg(p.bias + n0 + j + 2);
                if (n0 + j + 3 < p.N) o.w += __ldg(p.bias + n0 + j + 3);
              }
              *reinterpret_cast<float4*>(buf + sw128_offset(lane, j >> 2)) = o;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (p.flags & SB_GEMM_ACCUMULATE)
                asm volatile(
                    "cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group"
                    " [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_c)),
                    "r"(smem_u32(buf)), "r"(n0), "r"(m0)
                    : "memory");
              else
                asm volatile(
                    "cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group"
                    " [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_c)),
                    "r"(smem_u32(buf)), "r"(n0), "r"(m0)
                    : "memory");
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            ++out_slot;
          }
        } else if (row_ok && has_k && n0 < p.N) {
          if (p.flags & SB_GEMM_ACCUMULATE) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = n0 + j;
              if (n < p.N) {
                float x = __uint_as_float(v[j]);
                if (add_bias) x += __ldg(p.bias + n);
                atomicAdd(crow + n, x);
              }
            }
          } else if (vec_ok && n0 + 32 <= p.N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o;
              o.x = __uint_as_float(v[j + 0]);
              o.y = __uint_as_float(v[j + 1]);
              o.z = __uint_as_float(v[j + 2]);
              o.w = __uint_as_float(v[j + 3]);
              if (add_bias) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + j));
                o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
              }
              *reinterpret_cast<float4*>(crow + n0 + j) = o;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = n0 + j;
              if (n < p.N) {
                float x = __uint_as_float(v[j]);
                if (add_bias) x += __ldg(p.bias + n);
                crow[n] = x;
              }
            }
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
    }
    // all bulk stores of this thread must have completed before the CTA exits
    if (p.tma_store && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ----------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): the two CTAs of a cluster compute one 256 x 256 tile.
// Each CTA stages ITS 128 rows of A and ITS 128 rows of B; the pair's tensor cores read the B
// halves from both shared memories, so per CTA and k-block the shared-memory traffic is
// 16 KB written by TMA + 16 KB read by the MMA for 128x256x64 MACs, against 24 + 24 KB in the
// single-CTA 128x256 tile - the single-CTA tile is bounded by shared-memory bandwidth
// (~192 B/clk needed, 128 B/clk available => <= 67 % tensor utilisation, 55 % measured).
//   * rank 0 (leader) issues every MMA; both CTAs run a TMA producer whose loads signal the
//     LEADER's full barrier (cp.async.bulk.tensor.cta_group::2)
//   * tcgen05.commit.multicast frees the smem slot in both CTAs and publishes the accumulator to
//     both epilogues; the epilogues of both CTAs arrive on the leader's tmem-empty barrier
// ----------------------------------------------------------------------------------------------
SB_DEVINL uint32_t cta_rank_in_cluster() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
SB_DEVINL void cluster_barrier_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
SB_DEVINL uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
SB_DEVINL void tma_load_2d_pair(void* smem_dst, const void* tmap, uint32_t leader_bar, int32_t c0,
                                int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar),
        "r"(c0), "r"(c1)
      : "memory");
}
SB_DEVINL void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
SB_DEVINL void umma_commit_pair(uint64_t* bar) {   // arrives at this offset in BOTH CTAs
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64"
      " [%0], %1;" ::"r"(smem_u32(bar)), "h"((uint16_t)3)
      : "memory");
}
SB_DEVINL void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
SB_DEVINL void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0, ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!ok && ++spins > SB_SPIN_LIMIT) __trap();
  }
}

// Work distribution of the pair kernel: work item = (output tile, K split), round-robin over the
// CTA pairs, so that the pairs of one wave walk the same k range together (L2 reuse of the panels).
struct PairSched {
  int w, step, total_work, tiles_mn, kbt, kb_per_split;
  __device__ PairSched(const GemmParams& p, int pair_id, int n_pairs) {
    tiles_mn = p.m_tiles * p.n_tiles;
    kbt = p.k_blocks_total;
    total_work = tiles_mn * p.split_k;
    kb_per_split = (kbt + p.split_k - 1) / p.split_k;
    w = pair_id;
    step = n_pairs;
  }
  // next piece of work: output tile index and k-block range [kb0, kb1)
  __device__ bool next(int& tile, int& kb0, int& kb1) {
    if (w >= total_work) return false;
    const int split = w / tiles_mn;
    tile = w - split * tiles_mn;
    kb0 = split * kb_per_split;
    kb1 = kb0 + kb_per_split;
    if (kb1 > kbt) kb1 = kbt;
    w += step;
    return true;
  }
};

struct GemmPairCfg {
  static constexpr int BN = 256;                              // N of the pair's tile
  static constexpr int kStageBytes = (BM + BN / 2) * BK * 2;  // per CTA: 16 KB A + 16 KB B
  static constexpr int kStages = 6;
  static constexpr int kTmemCols = 512;                       // 2 accumulator stages x 256
  static constexpr int kStageOutBytes = 4 * 2 * 4096;
  static constexpr int kSmemBytes = kStages * kStageBytes + kStageOutBytes + 1024 + 256;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(192, 1)
gemm_bf16_tn_pair_kernel(const __grid_constant__ CUtensorMap tmap_a,
                         const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ CUtensorMap tmap_c, const GemmParams p) {
  using Cfg = GemmPairCfg;
  constexpr int kStages = Cfg::kStages;
  constexpr int BN = Cfg::BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~static_cast<uintptr_t>(1023));
  uint8_t* out_stage = tiles + kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(out_stage + Cfg::kStageOutBytes);
  uint64_t* full_bar = bars;                      // [kStages]  (the leader's are used)
  uint64_t* empty_bar = bars + kStages;           // [kStages]
  uint64_t* tfull_bar = bars + 2 * kStages;       // [2]
  uint64_t* tempty_bar = bars + 2 * kStages + 2;  // [2]        (the leader's are used)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cta_rank_in_cluster();
  const int pair_id = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_c);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 8);   // 4 epilogue warps x 2 CTAs
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"((uint32_t)Cfg::kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_barrier_all();   // the peer's barriers exist before anything signals them
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  PairSched sched(p, pair_id, n_pairs);           // p.m_tiles counts 256-row pair tiles here
  int tile, kb0, kb1;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      while (sched.next(tile, kb0, kb1)) {
        const int m_blk = tile / p.n_tiles;
        const int n_blk = tile - m_blk * p.n_tiles;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = tiles + stage * Cfg::kStageBytes;
          uint8_t* sb_ = sa + BM * BK * 2;
          const uint32_t lbar = map_to_cta(smem_u32(&full_bar[stage]), 0);
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
          if (p.a_mn) {
#pragma unroll
            for (int b = 0; b < BM / 64; ++b)
              tma_load_2d_pair(sa + b * MN_BOX_BYTES, &tmap_a, lbar,
                               m_blk * (2 * BM) + (int)rank * BM + b * 64, kb * BK);
          } else {
            tma_load_2d_pair(sa, &tmap_a, lbar, kb * BK, m_blk * (2 * BM) + (int)rank * BM);
          }
          if (p.b_mn) {
#pragma unroll
            for (int b = 0; b < BN / 2 / 64; ++b)
              tma_load_2d_pair(sb_ + b * MN_BOX_BYTES, &tmap_b, lbar,
                               n_blk * BN + (int)rank * (BN / 2) + b * 64, kb * BK);
          } else {
            tma_load_2d_pair(sb_, &tmap_b, lbar, kb * BK, n_blk * BN + (int)rank * (BN / 2));
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (rank == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(2 * BM, BN) | (p.a_mn ? (1u << 15) : 0u) |
                             (p.b_mn ? (1u << 16) : 0u);
      const uint64_t a_step = p.a_mn ? (uint64_t)(MN_KADV >> 4) : 2u;
      const uint64_t b_step = p.b_mn ? (uint64_t)(MN_KADV >> 4) : 2u;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      while (sched.next(tile, kb0, kb1)) {
        if (lane == 0) mbar_wait_cluster(&tempty_bar[acc], acc_phase ^ 1);
        __syncwarp();
        tc_fence_after_sync();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          if (lane == 0) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after_sync();
            const uint32_t sa = smem_u32(tiles + stage * Cfg::kStageBytes);
            const uint64_t da = p.a_mn ? umma_desc_sw128_mnmajor(sa) : umma_desc_sw128_kmajor(sa);
            const uint64_t db = p.b_mn ? umma_desc_sw128_mnmajor(sa + BM * BK * 2)
                                       : umma_desc_sw128_kmajor(sa + BM * BK * 2);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_bf16_ss_pair(tmem_d, da + a_step * k, db + b_step * k, idesc,
                                (kb > kb0 || k > 0) ? 1u : 0u);
            umma_commit_pair(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit_pair(&tfull_bar[acc]);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (kb1 <= kb0 && lane == 0) umma_commit_pair(&tfull_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue warps (2..5, both CTAs) =====================
    const int sub = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    unsigned int out_slot = 0;
    while (sched.next(tile, kb0, kb1)) {
      const int m_blk = tile / p.n_tiles;
      const int n_blk = tile - m_blk * p.n_tiles;
      const bool has_k = kb0 < kb1;
      const bool add_bias = (p.bias != nullptr) && (kb0 == 0);
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after_sync();
      const int m0 = m_blk * (2 * BM) + (int)rank * BM + sub * 32;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(sub * 32) << 16) + acc * BN + c * 32, v);
        tmem_ld_wait();
        const int n0 = n_blk * BN + c * 32;
        if (has_k && n0 < p.N && m0 < p.M) {      // warp-uniform
          uint8_t* buf = out_stage + ((warp - 2) * 2 + (out_slot & 1)) * 4096;
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o;
            o.x = __uint_as_float(v[j + 0]);
            o.y = __uint_as_float(v[j + 1]);
            o.z = __uint_as_float(v[j + 2]);
            o.w = __uint_as_float(v[j + 3]);
            if (add_bias) {
              if (n0 + j + 0 < p.N) o.x += __ldg(p.bias + n0 + j + 0);
              if (n0 + j + 1 < p.N) o.y += __ldg(p.bias + n0 + j + 1);
              if (n0 + j + 2 < p.N) o.z += __ldg(p.bias + n0 + j + 2);
              if (n0 + j + 3 < p.N) o.w += __ldg(p.bias + n0 + j + 3);
            }
            *reinterpret_cast<float4*>(buf + sw128_offset(lane, j >> 2)) = o;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (p.flags & SB_GEMM_ACCUMULATE)
              asm volatile(
                  "cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group"
                  " [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_c)),
                  "r"(smem_u32(buf)), "r"(n0), "r"(m0)
                  : "memory");
            else
              asm volatile(
                  "cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group"
                  " [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmap_c)),
                  "r"(smem_u32(buf)), "r"(n0), "r"(m0)
                  : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          ++out_slot;
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tempty_bar[acc]), 0));
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_barrier_all();   // neither CTA leaves while the pair's MMAs / remote arrives are in flight
  if (warp == 1) {
    tc_fence_after_sync();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)Cfg::kTmemCols)
                 : "memory");
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  return fn;
}

// 2-D bf16 tensor map over a row-major [rows, cols] matrix with leading dimension ld (elements);
// box = 64 columns x box_rows rows, SWIZZLE_128B, out-of-bounds reads return zero.
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, long long rows, long long cols,
                      long long ld, int box_rows) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return SB_ERR_CUDA;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ((ld * 2) & 15) != 0) return SB_ERR_INVALID;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? SB_OK : SB_ERR_CUDA;
}

int device_sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

// f32 tensor map over C [M][N] (ld = ldc): box 32 x 32, SWIZZLE_128B; stores clip at the edges
static int make_tmap_f32_c(CUtensorMap* map, float* base, long long rows, long long cols,
                           long long ld) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return SB_ERR_CUDA;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? SB_OK : SB_ERR_CUDA;
}

template <int BN>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, GemmParams p,
                       cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes);
    if (e != cudaSuccess) return SB_ERR_CUDA;
    attr_set = true;
  }
  p.n_tiles = (p.N + BN - 1) / BN;
  const int total = p.m_tiles * p.n_tiles * p.split_k;
  int grid = device_sm_count();
  if (grid > total) grid = total;
  CUtensorMap tc = ta;   // placeholder when the register epilogue is used
  p.tma_store = 0;
  if (!(p.flags & SB_GEMM_ROW_REMAP) && (p.ldc & 3) == 0 &&
      (reinterpret_cast<uintptr_t>(p.C) & 15) == 0) {
    if (make_tmap_f32_c(&tc, p.C, p.M, p.N, p.ldc) == SB_OK) p.tma_store = 1;
  }
  gemm_bf16_tn_kernel<BN><<<grid, 192, Cfg::kSmemBytes, stream>>>(ta, tb, tc, p);
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}

// K split of an ACCUMULATING GEMM (the caller's value is only a hint).  Work items = tiles x
// splits are dealt round-robin to `units` CTAs (or CTA pairs), so the launch takes
// ceil(tiles*split/units) rounds of (k-blocks per item + E) each, E ~ the epilogue / reduce-add
// pass of an item expressed in k-block times.  The minimum of that product fills whole waves -
// the dW_ih GEMM has 192 pair tiles for 74 pairs: 2.6 waves unsplit (3 rounds of 250 k-blocks),
// 12.97 waves with 5 splits (13 rounds of 50) - while every wave still walks K in lockstep, which
// keeps the operand panels in L2.  (A contiguous tiles x k-blocks "stream-K" partition was
// measured HBM-bound instead: 2.5 GB of DRAM reads for 0.26 GB of operands, no reuse.)
static int pick_wave_filling_split(long long tiles, int units, int k_blocks) {
  const long long kEpilogue = 4;
  int best_split = 1;
  long long best = -1;
  for (int sp = 1; sp <= 512; ++sp) {
    if (sp > 1 && k_blocks / sp < 8) break;
    const long long rounds = (tiles * sp + units - 1) / units;
    const long long cost = rounds * ((k_blocks + sp - 1) / sp + kEpilogue);
    if (best < 0 || cost < best) { best = cost; best_split = sp; }   // ties: fewer splits
  }
  return best_split;
}

// CTA-pair launch: needs the TMA-store epilogue (no row remap, 16-byte aligned C rows)
static int launch_gemm_pair(const CUtensorMap& ta, const CUtensorMap& tb, GemmParams p,
                            cudaStream_t stream) {
  using Cfg = GemmPairCfg;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes);
    if (e != cudaSuccess) return SB_ERR_CUDA;
    attr_set = true;
  }
  p.m_tiles = (p.M + 2 * BM - 1) / (2 * BM);
  p.n_tiles = (p.N + Cfg::BN - 1) / Cfg::BN;
  const int total = p.m_tiles * p.n_tiles * p.split_k;
  int pairs = device_sm_count() / 2;
  if (pairs > total) pairs = total;
  CUtensorMap tc;
  if (make_tmap_f32_c(&tc, p.C, p.M, p.N, p.ldc) != SB_OK) return SB_ERR_CUDA;
  p.tma_store = 1;
  gemm_bf16_tn_pair_kernel<<<2 * pairs, 192, Cfg::kSmemBytes, stream>>>(ta, tb, tc, p);
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}

}  // namespace sb

using namespace sb;

extern "C" int sb_gemm_bf16_tn(const void* A, long long lda, const void* B, long long ldb, float* C,
                               long long ldc, const float* bias, int M, int N, int K, int flags,
                               int split_k, int remap_B, int remap_T, int valid_B,
                               void* stream_) {
  if (!A || !B || !C || M <= 0 || N <= 0 || K <= 0) return SB_ERR_INVALID;
  if (split_k < 1) split_k = 1;
  if (split_k > 1 && !(flags & SB_GEMM_ACCUMULATE)) return SB_ERR_INVALID;
  if ((flags & SB_GEMM_ROW_REMAP) && (remap_B <= 0 || remap_T <= 0)) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  GemmParams p;
  p.C = C; p.bias = bias; p.ldc = ldc; p.M = M; p.N = N; p.K = K;
  p.k_blocks_total = (K + BK - 1) / BK;
  if (split_k > p.k_blocks_total) split_k = p.k_blocks_total;
  p.split_k = split_k; p.flags = flags;
  p.remap_B = remap_B; p.remap_T = remap_T; p.valid_B = valid_B;
  p.m_tiles = (M + BM - 1) / BM;
  p.n_tiles = 0;
  p.a_mn = (flags & SB_GEMM_A_MN) ? 1 : 0;
  p.b_mn = (flags & SB_GEMM_B_MN) ? 1 : 0;
  // tensor maps: K-major operands are [rows][K] with box {64 K, rows}; MN-major operands are
  // [K][rows] with box {64 rows, 64 K}
  auto tmap_a = [&](CUtensorMap* m, int box_rows) {
    return p.a_mn ? make_tmap_bf16_2d(m, A, K, M, lda, 64) : make_tmap_bf16_2d(m, A, M, K, lda, box_rows);
  };
  auto tmap_b = [&](CUtensorMap* m, int box_rows) {
    return p.b_mn ? make_tmap_bf16_2d(m, B, K, N, ldb, 64) : make_tmap_bf16_2d(m, B, N, K, ldb, box_rows);
  };

  // tile-N choice: the widest tile that still leaves >= ~1 wave of work
  const int sms = device_sm_count();
  int bn;
  if (N <= 32 && !p.b_mn) bn = 32;   // (an MN-major B tile is made of 64-wide boxes)
  else if (N <= 64) bn = 64;
  else if (N <= 128) bn = 128;
  else {
    const long long tiles256 = (long long)p.m_tiles * ((N + 255) / 256) * split_k;
    bn = (tiles256 >= sms || N > 2048) ? 256 : 128;
  }
  if (N > 128 && !(flags & SB_GEMM_ROW_REMAP) &&
      (ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
    const long long pair_tiles = (long long)((M + 2 * BM - 1) / (2 * BM)) * ((N + 255) / 256);
    const int pairs = sms / 2;
    int pair_split = split_k;
    if (flags & SB_GEMM_ACCUMULATE)
      pair_split = pick_wave_filling_split(pair_tiles, pairs, p.k_blocks_total);
    const bool use_pair = (flags & SB_GEMM_ACCUMULATE)
                              ? (pair_tiles * pair_split * 2 >= pairs)
                              : (bn == 256 && K >= 1024 && pair_tiles * split_k >= pairs);
    if (use_pair) {
      p.split_k = pair_split;
      CUtensorMap pa, pb;
      int prc = tmap_a(&pa, BM);
      if (prc != SB_OK) return prc;
      prc = tmap_b(&pb, 128);
      if (prc != SB_OK) return prc;
      return launch_gemm_pair(pa, pb, p, stream);
    }
  }
  if (flags & SB_GEMM_ACCUMULATE)
    p.split_k = pick_wave_filling_split((long long)p.m_tiles * ((N + bn - 1) / bn), sms,
                                        p.k_blocks_total);
  CUtensorMap ta, tb;
  int rc = tmap_a(&ta, BM);
  if (rc != SB_OK) return rc;
  rc = tmap_b(&tb, bn);
  if (rc != SB_OK) return rc;
  switch (bn) {
    case 32: return launch_gemm<32>(ta, tb, p, stream);
    case 64: return launch_gemm<64>(ta, tb, p, stream);
    case 128: return launch_gemm<128>(ta, tb, p, stream);
    default: return launch_gemm<256>(ta, tb, p, stream);
  }
}
