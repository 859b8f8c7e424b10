// Persistent GRU recurrence kernels (forward and backward in time) for sm_100a.
//
// Replaces the cuDNN RNN reached through nn.GRU in the reference encoder
// (speech/models/model.py:35-39 construction, :73 call; gate order r,z,n; bidirectional halves
// are summed by the caller, model.py:75-77) and the pred-net GRU of the transducer
// (speech/models/transducer_model.py:23-26,68).
//
// The time-batched input projection gi = X W_ih^T + b_ih is done for all T at once by
// sb_gemm_bf16_tn; these kernels run the T-serial part.  One launch per layer covers BOTH
// directions.  CTA c of direction d does the gate math of 16 hidden units, and the CTAs of a
// direction meet once per step at a grid barrier (one red.release.gpu + ld.acquire.gpu polling on a
// global counter).  Six kernels, three per direction of time:
//   * gru_fwd_kernel / gru_bwd_kernel (full gather): every CTA gathers ALL of h_{t-1} (backward:
//     the pre-activation gradients dgh_t, batch x 3H) through a ring of shared-memory slots, with
//     TMA multicast inside clusters of up to 4.  Any H % 16 == 0, up to 128 batch rows.
//   * gru_fwd_ks_kernel / gru_bwd_ks_kernel (K split): the 4 CTAs of a cluster jointly own 64
//     units; CTA r contracts only the r-th quarter of K into a batch-major accumulator, and the
//     partial products are reduce-scattered through distributed shared memory.  H % 256 == 0.
//   * gru_fwd_kt_kernel<UPT> / gru_bwd_kt_kernel (K split, transposed accumulator): the same
//     partition with the weights as the M-side operand, for small batches.
// All six have the same warp roles (warps 0..7 epilogue: TMEM -> gate math -> publish -> off-path
// stores; warp 8 MMA issuer and TMEM owner; warp 9 TMA producer) and share what is written once
// below: the shared-memory layout of each family (GruSmemLayout, which the kernels carve and the
// host sizes the launch from), setup and teardown, the per-thread loads and stores of UPT units,
// the gate math of each direction with its publish and off-path stores, and the K-split gather
// and MMA of each direction.  What differs is the exchange and the accumulator layout.
//
// Roofline: tensor work, but each step is bound by the all-gather + barrier latency; DESIGN.md
// reports us/step next to the tensor-pipe share.
#include "common.cuh"
#include <cuda.h>
#include <string.h>
#include <algorithm>

#include "../../include/speech_b200.h"

namespace sb {

static constexpr int GRU_HC = 16;            // hidden units per CTA
static constexpr int GRU_UPT = 8;            // hidden units per epilogue thread (batch-major)
static constexpr int GRU_MAX_RING = 16;      // smem ring slots for the gathered operand
static constexpr int GRU_EPI = 256;          // warps 0..7: epilogue
static constexpr int GRU_THREADS = GRU_EPI + 64;  // + warp 8: MMA issuer/TMEM owner, warp 9: TMA
static constexpr int KS = 4;                 // K split: CTAs of a cluster, quarters of K
static constexpr int GRU_KS_BWD_GROUPS = 4;  // K split, backward: full barriers (chunk groups)

typedef __nv_bfloat16 bf16;

struct GruFwdParams {
  const float* gi;     // [T*Bp][ndir*3H]  input projections (b_ih already added)
  const bf16* whh;     // [ndir][3H][H]    recurrent weights, bf16
  const float* bhh;    // [ndir][3H]
  float* y;            // [T*Bp][ndir*H]   h_t fp32
  bf16* xn;            // [T*Bp][ndir*H]   h_t bf16 (operand of the next projection)
  float* gates;        // [T*Bp][ndir][4][H] saved r,z,n,hn for backward ; may be null
  unsigned int* barrier;  // [ndir] zero-initialised counters
  unsigned long long* dbg;  // optional timeline (CTA 0): [step][16] globaltimer stamps, or null
  int T, Bp, H, ndir, ring, gc;   // ring: slots (groups of gc chunks) in shared memory
};

struct GruBwdParams {
  const float* dy;     // [T*Bp][ndir*H]   gradient w.r.t. this layer's output
  const float* y;      // [T*Bp][ndir*H]   forward h_t (fp32)
  const float* gates;  // [T*Bp][ndir][4][H]
  const bf16* whh;     // [ndir][3H][H]    W_hh as stored, bf16 (transposed while staging)
  bf16* dgi;           // [T*Bp][ndir*3H]  d(pre-activation) of the input projection, bf16
  bf16* dghn;          // [T*Bp][ndir*H]   dn_pre * r, token-major (wgrad of W_hn)
  bf16* xchg;          // [ndir][2][Bp][3H] per-step exchange of dgh_t (double-buffered)
  float* dbih;         // [ndir*3H] += sum_{t,b} dgi
  float* dbhh;         // [ndir*3H] += sum_{t,b} dgh
  unsigned int* barrier;  // [ndir]
  unsigned long long* dbg;
  int T, Bp, H, ndir, ring, gc;
};

// =============================================================================================
// shared-memory layout
// =============================================================================================
// One layout per kernel family.  The kernel carves its shared memory from it and the host requests
// `bytes` and decides from it whether the kernel fits, so the two cannot disagree.  Offsets are in
// bytes from the 1024-aligned base of dynamic shared memory; the gather ring starts at 0, and
// everything below `full` is zeroed at setup.
struct GruSmemLayout {
  int wtile;      // resident weight chunks (wrows x 64 bf16 each, K-major SWIZZLE_128B)
  int recv;       // K split: partial products received from the peers
  int stage;      // K split: partial products staged for the peers
  int full;       // `nfull` mbarriers: gathered chunks landed
  int nfull;
  int empty;      // full gather: GRU_MAX_RING mbarriers, ring slot free (0 = none)
  int accfull;    // mbarrier: accumulator complete
  int recvbar;    // K split: mbarrier, the peers' slices landed (0 = none)
  int tmem_slot;  // TMEM base address written by tcgen05.alloc
  int scratch;    // b_hh of the CTA's units (forward); bias-gradient reduction (full-gather bwd)
  int bytes;      // dynamic shared memory to request (alignment slack and reserved tail included)
};

__host__ __device__ __forceinline__ int gru_imax(int a, int b) { return a > b ? a : b; }

// Chunks of the gathered operand share one mbarrier per group of gc: the largest of 4, 3, 2, 1
// that divides nchunks.
__host__ __device__ __forceinline__ int gru_group_chunks(int nchunks) {
  return nchunks % 4 == 0 ? 4 : (nchunks % 3 == 0 ? 3 : (nchunks % 2 == 0 ? 2 : 1));
}

// Full gather: ring | weights | barriers | scratch.  The 128-row MMA read of the last ring slot
// overruns by (16 KB - Bp*128) into the weight region, which is padded to cover it.
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_full(int Bp, int nchunks, int wrows,
                                                                 int ring_bytes) {
  GruSmemLayout L;
  L.wtile = ring_bytes;
  L.full = L.wtile + gru_imax(nchunks * wrows * 128, 16384 - Bp * 128);
  L.recv = L.stage = L.full;
  L.nfull = GRU_MAX_RING;
  L.empty = L.full + GRU_MAX_RING * 8;
  L.accfull = L.empty + GRU_MAX_RING * 8;
  L.recvbar = 0;
  L.tmem_slot = L.accfull + 8;
  L.scratch = L.tmem_slot + 8;
  L.bytes = 1024 + L.scratch + 64 * 4 + 64;
  return L;
}

// K split: the whole K quarter is resident (ring of nchunks slots) | weights | receive and staging
// buffers of the reduce-scatter (at least xchg_min bytes together) | barriers | `tail` bytes for
// the TMEM slot and the bias.
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_ksplit(int Bp, int nchunks, int wrows,
                                                                   int recv_bytes, int stage_bytes,
                                                                   int xchg_min, int nfull,
                                                                   int tail) {
  GruSmemLayout L;
  L.wtile = nchunks * Bp * 128;
  L.recv = L.wtile + nchunks * wrows * 128;
  L.stage = L.recv + recv_bytes;
  L.full = L.recv + gru_imax(recv_bytes + stage_bytes, xchg_min);
  L.nfull = nfull;
  L.empty = 0;
  L.accfull = L.full + nfull * 8;
  L.recvbar = L.accfull + 8;
  L.tmem_slot = L.recvbar + 8;
  L.scratch = L.tmem_slot + 8;
  L.bytes = 1024 + L.full + tail;
  return L;
}

// ks forward: 192 weight rows (gate x 64 units); [KS][Bp][48] floats received and staged.  The
// 128-row A read of the last chunk runs past the ring into the weights (finite, rows >= Bp unused).
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_fwd_ks(int Bp, int H) {
  const int xb = KS * Bp * 3 * GRU_HC * 4;
  return gru_layout_ksplit(Bp, H / KS / 64, 3 * KS * GRU_HC, xb, xb, 0, 1, 512);
}
// ks backward: 64 weight rows (units of W_hh^T); [KS][Bp][16] floats received and staged.
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_bwd_ks(int Bp, int H) {
  const int xb = KS * Bp * GRU_HC * 4;
  return gru_layout_ksplit(Bp, 3 * H / KS / 64, KS * GRU_HC, xb, xb, 0, GRU_KS_BWD_GROUPS, 256);
}
// kt forward: slices of [48][Bp+4] floats, KS received and KS-1 staged.  The N-side read of the
// last chunk runs up to 8 rows past the ring into the weights, and the 128-row M-side read of tile
// 1 runs 64 rows past its 64 valid ones (into the next chunk / the receive buffer): both only feed
// accumulator columns / lanes that are never read.
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_fwd_kt(int Bp, int H) {
  const int slice = 3 * GRU_HC * (Bp + 4) * 4;
  return gru_layout_ksplit(Bp, H / KS / 64, 3 * KS * GRU_HC, KS * slice, (KS - 1) * slice, 0, 1,
                           512);
}
// kt backward: slices of [16][Bp+4] floats.  The 128-row M-side read of the last weight chunk
// needs 8 KB after the weights, which the exchange buffers cover only for large batches.
__host__ __device__ __forceinline__ GruSmemLayout gru_layout_bwd_kt(int Bp, int H) {
  const int slice = GRU_HC * (Bp + 4) * 4;
  return gru_layout_ksplit(Bp, 3 * H / KS / 64, KS * GRU_HC, KS * slice, (KS - 1) * slice, 8192,
                           GRU_KS_BWD_GROUPS, 256);
}

struct GruSmem {
  uint8_t* ring;
  uint8_t* wtile;
  float* recv;
  float* stage;
  uint64_t* full;
  uint64_t* empty;
  uint64_t* accfull;
  uint64_t* recvbar;
  uint32_t* tmem_slot;
  float* scratch;
};

SB_DEVINL GruSmem gru_carve(uint8_t* raw, const GruSmemLayout& L) {
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  GruSmem s;
  s.ring = base;
  s.wtile = base + L.wtile;
  s.recv = reinterpret_cast<float*>(base + L.recv);
  s.stage = reinterpret_cast<float*>(base + L.stage);
  s.full = reinterpret_cast<uint64_t*>(base + L.full);
  s.empty = reinterpret_cast<uint64_t*>(base + L.empty);
  s.accfull = reinterpret_cast<uint64_t*>(base + L.accfull);
  s.recvbar = reinterpret_cast<uint64_t*>(base + L.recvbar);
  s.tmem_slot = reinterpret_cast<uint32_t*>(base + L.tmem_slot);
  s.scratch = reinterpret_cast<float*>(base + L.scratch);
  return s;
}

SB_DEVINL unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define GRU_STAMP(ev)                                                              \
  do {                                                                             \
    if (p.dbg && blockIdx.x == 0 && step < 64) p.dbg[step * 16 + (ev)] = gtime(); \
  } while (0)

// ---- per-direction grid barrier ------------------------------------------------------------
SB_DEVINL void grid_arrive(unsigned int* ctr) { red_release_gpu_add(ctr, 1u); }
// One ld.acquire.gpu per poll: its implied fence throttles the poll rate.  (Relaxed polling, with
// or without nanosleep, was measured SLOWER, 7.8 vs 7.3 us/step: the tight spin of 128 pollers on
// the counter's L2 line delays the arriving reductions.)
SB_DEVINL void grid_wait(const unsigned int* ctr, unsigned int target) {
  unsigned int spins = 0;
  while (ld_acquire_gpu(ctr) < target) {
    if (++spins > SB_SPIN_LIMIT) __trap();
  }
}
SB_DEVINL void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(GRU_EPI) : "memory"); }

// ---- cluster helpers ---------------------------------------------------------------------------
SB_DEVINL uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
SB_DEVINL uint32_t cluster_size() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
SB_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA box load multicast to every CTA in `mask` (same smem offset + same mbarrier offset in each)
SB_DEVINL void tma_load_2d_mc(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0,
                              int32_t c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
// arrive (when all prior MMAs of this thread retire) on the mbarrier at this offset in every CTA
// of `mask`
SB_DEVINL void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64"
      " [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
SB_DEVINL uint32_t mapa_shared(uint32_t local_addr, uint32_t peer) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(peer));
  return r;
}
// bulk copy from this CTA's shared memory into a PEER's shared memory (DSMEM through the copy
// engine), completing `bytes` on the peer's mbarrier.  Measured: pushing the reduce-scatter
// slices with per-thread st.shared::cluster took 4.1 us for 36 KB (~9 KB/us per SM).
SB_DEVINL void bulk_s2peer(uint32_t peer_dst, const void* local_src, uint32_t bytes,
                           uint32_t peer_bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(peer_dst), "r"(smem_u32(local_src)), "r"(bytes), "r"(peer_bar)
      : "memory");
}

// ---- setup and teardown -----------------------------------------------------------------------
// Zero the ring, weight and exchange regions (rows past the batch and columns past K must read as
// finite zeros), stage the resident operand (`stage`, which differs per kernel), initialise the
// barriers, allocate `tmem_cols` TMEM columns, and make all of it visible to the async proxy and to
// the peer CTAs before any of them multicasts or copies into this CTA.  The empty barriers of the
// full gather count one arrive per CTA of the cluster (`cluster_ctas`).  Returns the TMEM base.
template <class Stage>
SB_DEVINL uint32_t gru_setup(const GruSmem& s, const GruSmemLayout& L, const CUtensorMap* tm,
                             uint32_t tmem_cols, uint32_t cluster_ctas, Stage stage) {
  const int tid = threadIdx.x;
  for (int k = tid; k < L.full / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(s.ring)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  stage();
  if (tid == 0) {
    for (int i = 0; i < L.nfull; ++i) {
      mbar_init(&s.full[i], 1);
      if (L.empty) mbar_init(&s.empty[i], cluster_ctas);
    }
    mbar_init(s.accfull, 1);
    // one local arrive.expect_tx per step; the peers' copies complete_tx
    if (L.recvbar) mbar_init(s.recvbar, 1);
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if ((tid >> 5) == 8) tmem_alloc(s.tmem_slot, tmem_cols);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();   // peers' barriers are initialised before anyone multicasts into them
  return *s.tmem_slot;
}

SB_DEVINL void gru_teardown(uint32_t tmem_base, uint32_t tmem_cols) {
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while peers may still signal its barriers
  if ((threadIdx.x >> 5) == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// =============================================================================================
// full gather: ring of gathered chunks
// =============================================================================================
// The gathered operand of one step is `nchunks` [Bp x 64] boxes, handled in groups of `gc` chunks
// that share ONE full/empty mbarrier pair (an mbarrier wait costs ~100 ns even when it is already
// complete, so per-chunk barriers were 3 us of a 10 us step).  Group g uses ring slot g % ring and
// ngroups % ring == 0, so every slot is used upr = ngroups/ring times per step and the mbarrier
// phase of use (k, g) is k*upr + g/ring for both barriers of the slot.
//
// TMA producer (one thread per CTA).  Every CTA arms its own full barriers; chunk c is fetched
// by the CTA whose cluster rank is c % CS and multicast to the whole cluster.
SB_DEVINL void tma_gather(const GruSmem& s, const CUtensorMap* tm, int row0, int Bp, int nchunks,
                          int ring, int gc, int k, uint32_t rank, uint32_t cs) {
  const int stride = Bp * 128;
  const int ngroups = nchunks / gc;
  const int upr = ngroups / ring;
  const uint16_t mask = (uint16_t)((1u << cs) - 1u);
  for (int g = 0; g < ngroups; ++g) {
    const int slot = g % ring;
    const unsigned int P = (unsigned int)(k * upr + g / ring);
    if (g >= ring) mbar_wait(&s.empty[slot], (P - 1u) & 1u);   // released by ALL CTAs of the cluster
    mbar_expect_tx(&s.full[slot], (uint32_t)(stride * gc));
    for (int i = 0; i < gc; ++i) {
      const int c = g * gc + i;
      if ((uint32_t)c % cs != rank) continue;
      uint8_t* dst = s.ring + (slot * gc + i) * stride;
      if (cs > 1) tma_load_2d_mc(dst, tm, &s.full[slot], c * 64, row0, mask);
      else tma_load_2d(dst, tm, &s.full[slot], c * 64, row0);
    }
  }
}

// MMA thread: consume the step's chunks against the resident weight chunks.
template <int N>
SB_DEVINL void mma_consume(const GruSmem& s, uint32_t tmem_d, int nchunks, int wchunk_bytes,
                           int Bp, int ring, int gc, int k, uint32_t cs) {
  constexpr uint32_t idesc = umma_idesc_bf16_f32(128, N);
  const int stride = Bp * 128;
  const int ngroups = nchunks / gc;
  const int upr = ngroups / ring;
  const uint16_t mask = (uint16_t)((1u << cs) - 1u);
  for (int g = 0; g < ngroups; ++g) {
    const int slot = g % ring;
    const unsigned int P = (unsigned int)(k * upr + g / ring);
    mbar_wait(&s.full[slot], P & 1u);
    tc_fence_after_sync();
    for (int i = 0; i < gc; ++i) {
      const int c = g * gc + i;
      const uint64_t da = umma_desc_sw128_kmajor(smem_u32(s.ring + (slot * gc + i) * stride));
      const uint64_t db = umma_desc_sw128_kmajor(smem_u32(s.wtile + c * wchunk_bytes));
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
        umma_bf16_ss(tmem_d, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                     (c > 0 || kk > 0) ? 1u : 0u);
    }
    if (ring < ngroups) {
      if (cs > 1) umma_commit_mc(&s.empty[slot], mask);
      else umma_commit(&s.empty[slot]);
    }
  }
  umma_commit(s.accfull);
}

// =============================================================================================
// K split: one step of the gather and of the product, per direction
// =============================================================================================
// Forward: the CTA's K quarter of h_{t-1} (columns col0.., rows row0.. of xn) stays resident
// whole, behind ONE full barrier.
SB_DEVINL void ks_gather_fwd(const GruSmem& s, const CUtensorMap* tm, int stride, int nchunks,
                             int col0, int row0) {
  mbar_expect_tx(s.full, (uint32_t)(stride * nchunks));
  for (int c = 0; c < nchunks; ++c)
    tma_load_2d(s.ring + c * stride, tm, s.full, col0 + c * 64, row0);
}
// Batch-major (ks): D[batch x 192] = h * W^T.  Transposed (kt): D0[128 x NB] = W(r,z rows) * h^T
// at TMEM column 0 and D1 = W(n rows) * h^T at column 64, the weight chunk being the M-side
// operand and `idesc` of N = NB.
SB_DEVINL void ks_mma_fwd(const GruSmem& s, uint32_t tmem, int stride, int nchunks, int wchunk,
                          uint32_t idesc, bool transposed, uint32_t parity) {
  mbar_wait(s.full, parity);
  tc_fence_after_sync();
  for (int c = 0; c < nchunks; ++c) {
    const uint64_t dh = umma_desc_sw128_kmajor(smem_u32(s.ring + c * stride));
    const uint64_t dw = umma_desc_sw128_kmajor(smem_u32(s.wtile + c * wchunk));
    if (!transposed) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
        umma_bf16_ss(tmem, dh + (uint64_t)(kk * 2), dw + (uint64_t)(kk * 2), idesc,
                     (c > 0 || kk > 0) ? 1u : 0u);
    } else {
      const uint64_t dw1 = umma_desc_sw128_kmajor(smem_u32(s.wtile + c * wchunk + 128 * 128));
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
        umma_bf16_ss(tmem, dw + (uint64_t)(kk * 2), dh + (uint64_t)(kk * 2), idesc, acc);
        umma_bf16_ss(tmem + 64, dw1 + (uint64_t)(kk * 2), dh + (uint64_t)(kk * 2), idesc, acc);
      }
    }
  }
  umma_commit(s.accfull);
}

// Backward: the CTA's K quarter of dgh_t (3H/4 columns) in groups of gc chunks, one full barrier
// per group (at most GRU_KS_BWD_GROUPS groups; the host checks).
SB_DEVINL void ks_gather_bwd(const GruSmem& s, const CUtensorMap* tm, int stride, int ngroups,
                             int gc, int col0, int row0) {
  for (int g = 0; g < ngroups; ++g) {
    mbar_expect_tx(&s.full[g], (uint32_t)(stride * gc));
    for (int i = 0; i < gc; ++i) {
      const int c = g * gc + i;
      tma_load_2d(s.ring + c * stride, tm, &s.full[g], col0 + c * 64, row0);
    }
  }
}
// Batch-major (ks): D[batch x 64 units] = dgh * W_hh.  Transposed (kt): D^T[64 units x NB], the
// weight chunk being the M-side operand.
SB_DEVINL void ks_mma_bwd(const GruSmem& s, uint32_t tmem, int stride, int ngroups, int gc,
                          int wchunk, uint32_t idesc, bool transposed, uint32_t parity) {
  for (int g = 0; g < ngroups; ++g) {
    mbar_wait(&s.full[g], parity);
    tc_fence_after_sync();
    for (int i = 0; i < gc; ++i) {
      const int c = g * gc + i;
      const uint64_t dh = umma_desc_sw128_kmajor(smem_u32(s.ring + c * stride));
      const uint64_t dw = umma_desc_sw128_kmajor(smem_u32(s.wtile + c * wchunk));
      const uint64_t da = transposed ? dw : dh, db = transposed ? dh : dw;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
        umma_bf16_ss(tmem, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                     (c > 0 || kk > 0) ? 1u : 0u);
    }
  }
  umma_commit(s.accfull);
}

// Backward staging of the K-split kernels: rows = the cluster's 64 units of W_hh^T (k0c..),
// columns = the CTA's K quarter.  W_hh is read as stored ([3H][H]: the cluster's 64 units are 128
// contiguous bytes of row k) and transposed on the way into shared memory.  The 64 rows are grouped
// by owner: rows 16q..16q+15 belong to CTA q of the cluster.
SB_DEVINL void ks_stage_whh_t(uint8_t* wtile, const bf16* whh, int H, int dir, int k0c,
                              uint32_t crank) {
  constexpr int WCHUNK = 64 * 128;
  const int K3 = 3 * H, KQ = K3 / KS;
  for (int k = threadIdx.x; k < KQ * 8; k += GRU_THREADS) {
    const int kl = k >> 3, piece = k & 7;       // local k, 8-unit piece of the 64 units
    const uint4 v = *reinterpret_cast<const uint4*>(
        whh + ((long long)dir * K3 + (long long)crank * KQ + kl) * H + k0c + piece * 8);
    const unsigned short* e = reinterpret_cast<const unsigned short*>(&v);
    uint8_t* chunk = wtile + (kl >> 6) * WCHUNK + (kl & 7) * 2;
#pragma unroll
    for (int q = 0; q < 8; ++q)
      *reinterpret_cast<unsigned short*>(
          chunk + sw128_offset((uint32_t)(piece * 8 + q), (uint32_t)((kl & 63) >> 3))) = e[q];
  }
}

// =============================================================================================
// per-thread work: UPT consecutive units of one batch row (8 batch-major, 1 or 2 in kt)
// =============================================================================================
SB_DEVINL float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
SB_DEVINL float fast_tanh(float x) {
  // 1 - 2/(exp(2x)+1), clamped so exp never overflows (__fdividef(2, inf) is not guaranteed 0)
  const float xc = fminf(fmaxf(x, -15.f), 15.f);
  return 1.0f - __fdividef(2.0f, __expf(2.0f * xc) + 1.0f);
}

SB_DEVINL uint4 pack8(const float (&v)[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
  return r;
}
// One-touch data (gi, saved gates, dy, fp32 state, GEMM operands written for later kernels) uses
// the streaming cache policy (.cs) so that it does not evict the latency-critical bf16 exchange
// buffers, which every CTA re-reads from L2 each step.
template <int UPT>
SB_DEVINL void ldu(const float* p, float (&v)[UPT]) {
  if constexpr (UPT == 8) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(p));
    const float4 b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else if constexpr (UPT == 2) {
    const float2 a = __ldcs(reinterpret_cast<const float2*>(p));
    v[0] = a.x; v[1] = a.y;
  } else {
    v[0] = __ldcs(p);
  }
}
template <int UPT>
SB_DEVINL void stu(float* p, const float (&v)[UPT]) {
  if constexpr (UPT == 8) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
    __stcs(reinterpret_cast<float4*>(p) + 1, make_float4(v[4], v[5], v[6], v[7]));
  } else if constexpr (UPT == 2) {
    __stcs(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
  } else {
    __stcs(p, v[0]);
  }
}
// the bf16 exchange, re-read by every CTA: default cache policy
template <int UPT>
SB_DEVINL void st_bf16u(bf16* p, const float (&v)[UPT]) {
  if constexpr (UPT == 8) {
    *reinterpret_cast<uint4*>(p) = pack8(v);
  } else if constexpr (UPT == 2) {
    *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(v[0], v[1]);
  } else {
    *p = __float2bfloat16_rn(v[0]);
  }
}
// bf16 operands of later GEMMs: streaming (the backward kernels run UPT = 8 or 1)
template <int UPT>
SB_DEVINL void st_stream_bf16u(bf16* p, const float (&v)[UPT]) {
  if constexpr (UPT == 8) {
    __stcs(reinterpret_cast<uint4*>(p), pack8(v));
  } else {
    static_assert(UPT == 1, "st_stream_bf16u: UPT 8 or 1");
    const unsigned short u = __bfloat16_as_ushort(__float2bfloat16_rn(v[0]));
    asm volatile("st.global.cs.u16 [%0], %1;" ::"l"(p), "h"(u) : "memory");
  }
}

SB_DEVINL void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7])
      : "r"(taddr)
      : "memory");
}

// Saved per step by the forward pass for the backward one: r, z, n and hn = W_hn h_{t-1} + b_hn.
template <int UPT>
struct GruGates {
  float r[UPT], z[UPT], n[UPT], hn[UPT];
};
// Backward per step: d(pre-activation) of r, z, n and dn * r (also used for their sums over t, b).
template <int UPT>
struct GruGrad {
  float r[UPT], z[UPT], n[UPT], nr[UPT];
};

// All epilogue threads have published: one arrive per CTA on the direction's grid barrier
// (release: cumulative over the CTA's writes ordered by bar.sync).
template <class Params>
SB_DEVINL void gru_arrive(const Params& p, int step, int tid, unsigned int* ctr, bool skew_probe) {
  epi_barrier();
  if (tid == 0) {
    GRU_STAMP(7);
    if (skew_probe && p.dbg && step == 20) p.dbg[1024 + blockIdx.x] = gtime();   // skew probe
    grid_arrive(ctr);
    GRU_STAMP(9);
  }
}

// ---- forward cell ---------------------------------------------------------------------------
// the input projections of step t do not depend on the recurrence: fetched first
template <int UPT>
SB_DEVINL void gru_load_gi(const GruFwdParams& p, int t, int row, int dir, int ju,
                           float (&gi)[3][UPT]) {
  const int H = p.H;
  const float* g = p.gi + ((long long)t * p.Bp + row) * (p.ndir * 3 * H) + dir * 3 * H + ju;
#pragma unroll
  for (int gg = 0; gg < 3; ++gg) ldu<UPT>(g + gg * H, gi[gg]);
}
template <int UPT>
SB_DEVINL void gru_cell_fwd(const float (&gi)[3][UPT], const float (&acc)[3][UPT],
                            const float (&bias)[3][UPT], float (&h)[UPT], GruGates<UPT>& g) {
#pragma unroll
  for (int jj = 0; jj < UPT; ++jj) {
    g.r[jj] = fast_sigmoid(gi[0][jj] + acc[0][jj] + bias[0][jj]);
    g.z[jj] = fast_sigmoid(gi[1][jj] + acc[1][jj] + bias[1][jj]);
    g.hn[jj] = acc[2][jj] + bias[2][jj];
    g.n[jj] = fast_tanh(gi[2][jj] + g.r[jj] * g.hn[jj]);
    h[jj] = (1.f - g.z[jj]) * g.n[jj] + g.z[jj] * h[jj];
  }
}
// critical path: only the bf16 h_t that the other CTAs gather next step (then gru_arrive)
template <int UPT>
SB_DEVINL void gru_publish_fwd(const GruFwdParams& p, int step, int tid, bool active, bf16* dst,
                               const float (&h)[UPT], unsigned int* ctr, bool skew_probe) {
  if (active) {
    st_bf16u<UPT>(dst, h);
    if (tid == 0) GRU_STAMP(5);
    fence_proxy_async_global();   // generic writes -> other CTAs' TMA reads
    if (tid == 0) GRU_STAMP(6);
  }
  gru_arrive(p, step, tid, ctr, skew_probe);
}
// off the critical path: fp32 state, saved gates
template <int UPT>
SB_DEVINL void gru_store_fwd(const GruFwdParams& p, long long m, int dir, int ju,
                             const float (&h)[UPT], const GruGates<UPT>& g) {
  const int H = p.H;
  stu<UPT>(p.y + m * (p.ndir * H) + dir * H + ju, h);
  if (p.gates) {
    float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
    stu<UPT>(go, g.r);
    stu<UPT>(go + H, g.z);
    stu<UPT>(go + 2 * H, g.n);
    stu<UPT>(go + 3 * H, g.hn);
  }
}

// ---- backward cell --------------------------------------------------------------------------
// saved activations of step t (row m), dL/dy and h_{t-1} (row mp): independent of the recurrence,
// fetched first
template <int UPT>
SB_DEVINL void gru_load_bwd(const GruBwdParams& p, long long m, long long mp, bool has_prev,
                            int dir, int ju, GruGates<UPT>& g, float (&dh)[UPT],
                            float (&hp)[UPT]) {
  const int H = p.H, D = p.ndir * H;
  const float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
  ldu<UPT>(go, g.r);
  ldu<UPT>(go + H, g.z);
  ldu<UPT>(go + 2 * H, g.n);
  ldu<UPT>(go + 3 * H, g.hn);
  ldu<UPT>(p.dy + m * D + dir * H + ju, dh);
  if (has_prev) {
    ldu<UPT>(p.y + mp * D + dir * H + ju, hp);
  } else {
#pragma unroll
    for (int jj = 0; jj < UPT; ++jj) hp[jj] = 0.f;
  }
}
// dh_rec: in, the part of dL/dh_t that arrived through the recurrence; out, the direct path
// h_{t-1} -> h_t (the W_hh path is added next step).
template <int UPT>
SB_DEVINL void gru_cell_bwd(const GruGates<UPT>& a, const float (&dh)[UPT], const float (&hp)[UPT],
                            float (&dh_rec)[UPT], GruGrad<UPT>& d, GruGrad<UPT>& db) {
#pragma unroll
  for (int jj = 0; jj < UPT; ++jj) {
    const float g = dh[jj] + dh_rec[jj];
    d.n[jj] = g * (1.f - a.z[jj]) * (1.f - a.n[jj] * a.n[jj]);
    d.z[jj] = g * (hp[jj] - a.n[jj]) * a.z[jj] * (1.f - a.z[jj]);
    d.r[jj] = d.n[jj] * a.hn[jj] * a.r[jj] * (1.f - a.r[jj]);
    d.nr[jj] = d.n[jj] * a.r[jj];
    dh_rec[jj] = g * a.z[jj];
    db.r[jj] += d.r[jj];
    db.z[jj] += d.z[jj];
    db.n[jj] += d.n[jj];
    db.nr[jj] += d.nr[jj];
  }
}
// critical path: the exchange row [dr | dz | dn*r] that every CTA gathers for the next product
// (x: this thread's units in row `row` of the step's exchange buffer; then gru_arrive)
template <int UPT>
SB_DEVINL void gru_publish_bwd(const GruBwdParams& p, int step, int tid, bool active, bf16* x,
                               const GruGrad<UPT>& d, unsigned int* ctr) {
  if (step + 1 < p.T) {   // the last step processed has no successor
    if (active) {
      st_bf16u<UPT>(x, d.r);
      st_bf16u<UPT>(x + p.H, d.z);
      st_bf16u<UPT>(x + 2 * p.H, d.nr);
      if (tid == 0) GRU_STAMP(5);
      fence_proxy_async_global();
      if (tid == 0) GRU_STAMP(6);
    }
    gru_arrive(p, step, tid, ctr, false);
  }
}
// off the critical path: operands of the dX / dW GEMMs
template <int UPT>
SB_DEVINL void gru_store_bwd(const GruBwdParams& p, long long m, int dir, int ju,
                             const GruGrad<UPT>& d) {
  const int H = p.H, K3 = 3 * H;
  bf16* o = p.dgi + m * (p.ndir * K3) + dir * K3 + ju;
  st_stream_bf16u<UPT>(o, d.r);
  st_stream_bf16u<UPT>(o + H, d.z);
  st_stream_bf16u<UPT>(o + 2 * H, d.n);
  st_stream_bf16u<UPT>(p.dghn + m * (p.ndir * H) + dir * H + ju, d.nr);
}

// =============================================================================================
// forward, full gather
//   * CTA c of direction d owns 16 hidden units j0..j0+15: its 48 rows of W_hh (r,z,n) stay
//     resident in shared memory (bf16, UMMA K-major SWIZZLE_128B chunks) for all T steps;
//   * per step every CTA needs ALL of h_{t-1} (bf16, written by the CTAs of its direction in the
//     previous step).  CTAs form thread-block clusters of up to 4; each CTA fetches 1/CS of the
//     [Bp x 64] chunks with TMA and MULTICASTS them into the shared memory of all CTAs of its
//     cluster, so L2 is read once per cluster instead of once per CTA (the un-multicast version
//     was bound by 64 SMs hammering the same L2 lines: 4 us of a 13 us step);
//   * one thread issues tcgen05.mma  D[batch(128) x 48] += h_{t-1}[batch x 64] * Wslice[48 x 64]^T
//     per chunk as its mbarrier completes; accumulators live in TMEM;
//   * 8 epilogue warps (thread = TMEM lane = batch row, 8 hidden units each) read the
//     accumulators with tcgen05.ld, apply the gate math in fp32 (h_{t-1} of the thread's own units
//     stays in registers across steps), publish the bf16 h_t, arrive on the per-direction grid
//     barrier, and only then write the fp32 state / saved gates.
// =============================================================================================
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_fwd_kernel(const __grid_constant__ CUtensorMap tm_d0, const __grid_constant__ CUtensorMap tm_d1,
               const GruFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int j0 = (blockIdx.x % nC) * GRU_HC;
  const int nchunks = (H + 63) / 64;
  constexpr int WCHUNK = 48 * 128;  // 48 rows x 64 bf16
  const GruSmemLayout L = gru_layout_full(Bp, nchunks, 48, p.ring * p.gc * Bp * 128);
  const GruSmem s = gru_carve(smem_raw, L);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const uint32_t crank = cluster_rank(), csize = cluster_size();

  const uint32_t tmem_base = gru_setup(s, L, tm, 64, csize, [&] {
    // the 48 weight rows (gate g, unit jj) and their b_hh
    const int pieces_per_row = nchunks * 8;
    for (int k = tid; k < 48 * pieces_per_row; k += GRU_THREADS) {
      const int r = k / pieces_per_row, pc = k % pieces_per_row;
      const int g = r / GRU_HC, jj = r % GRU_HC;
      const int col = pc * 8;
      if (col < H) {
        const uint4 v = *reinterpret_cast<const uint4*>(
            p.whh + ((long long)dir * 3 * H + g * H + j0 + jj) * H + col);
        *reinterpret_cast<uint4*>(s.wtile + (pc >> 3) * WCHUNK + sw128_offset(r, pc & 7)) = v;
      }
    }
    if (tid < 48) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      s.scratch[tid] = p.bhh[dir * 3 * H + g * H + j0 + jj];
    }
  });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      for (int step = 1; step < T; ++step) {
        const int t = dir == 0 ? step : (T - 1 - step);
        const int tp = dir == 0 ? t - 1 : t + 1;
        grid_wait(ctr, (unsigned int)nC * step);   // all CTAs published h_{tp}
        GRU_STAMP(0);
        // (the writers ran fence.proxy.async before their release; no reader-side proxy fence)
        tma_gather(s, tm, tp * Bp, Bp, nchunks, p.ring, p.gc, step - 1, crank, csize);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      for (int step = 1; step < T; ++step) {
        mma_consume<48>(s, tmem_base, nchunks, WCHUNK, Bp, p.ring, p.gc, step - 1, csize);
        GRU_STAMP(2);
      }
    }
  } else {
    // ===================== epilogue: thread = (batch row, half of the 16 units) ==============
    const int row = (warp & 3) * 32 + lane;      // TMEM lane this thread may read
    const int uh = warp >> 2;                    // which 8 of the CTA's 16 units
    const int ju = j0 + uh * GRU_UPT;
    float hprev[GRU_UPT];
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) hprev[jj] = 0.f;
    float bias[3][GRU_UPT];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int jj = 0; jj < GRU_UPT; ++jj) bias[g][jj] = s.scratch[g * 16 + uh * GRU_UPT + jj];
    const bool active = row < Bp;
    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? step : (T - 1 - step);
      float gi[3][GRU_UPT];
      if (active) gru_load_gi(p, t, row, dir, ju, gi);
      float acc[3][GRU_UPT];
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        uint32_t v[8];
#pragma unroll
        for (int gg = 0; gg < 3; ++gg) {
          tmem_ld_32x32b_x8(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + gg * 16 + uh * GRU_UPT,
                            v);
          tmem_ld_wait();
#pragma unroll
          for (int jj = 0; jj < GRU_UPT; ++jj) acc[gg][jj] = __uint_as_float(v[jj]);
        }
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
      } else {
#pragma unroll
        for (int gg = 0; gg < 3; ++gg)
#pragma unroll
          for (int jj = 0; jj < GRU_UPT; ++jj) acc[gg][jj] = 0.f;
      }
      const long long m = (long long)t * Bp + row;
      GruGates<GRU_UPT> g;
      if (active) gru_cell_fwd(gi, acc, bias, hprev, g);
      gru_publish_fwd(p, step, tid, active, p.xn + m * D + dir * H + ju, hprev, ctr, false);
      if (active) gru_store_fwd(p, m, dir, ju, hprev, g);
      if (tid == 0) GRU_STAMP(10);
    }
  }
  gru_teardown(tmem_base, 64);
}

// =============================================================================================
// backward, full gather (reverse of the forward time order of each direction): the structure of
// gru_fwd_kernel with W_hh^T resident (16 rows x 3H) and the all-gather over the pre-activation
// gradients dgh_t (batch x 3H).
// =============================================================================================
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_bwd_kernel(const __grid_constant__ CUtensorMap tm_d0, const __grid_constant__ CUtensorMap tm_d1,
               const GruBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int j0 = (blockIdx.x % nC) * GRU_HC;
  const int K3 = 3 * H;
  const int nchunks = (K3 + 63) / 64;
  constexpr int WCHUNK = 16 * 128;  // 16 rows x 64 bf16
  const GruSmemLayout L = gru_layout_full(Bp, nchunks, 16, p.ring * p.gc * Bp * 128);
  const GruSmem s = gru_carve(smem_raw, L);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const uint32_t crank = cluster_rank(), csize = cluster_size();

  const uint32_t tmem_base = gru_setup(s, L, tm, 32, csize, [&] {
    // resident operand: rows = the 16 hidden units j0..j0+15 of W_hh^T, K = 3H.  W_hh is read as
    // stored ([3H][H]: 32 contiguous bytes per k) and transposed on the way into shared memory
    for (int k = tid; k < K3 * 2; k += GRU_THREADS) {
      const int kk = k >> 1, half = k & 1;
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * K3 + kk) * H + j0 + half * 8);
      const unsigned short* e = reinterpret_cast<const unsigned short*>(&v);
      uint8_t* chunk = s.wtile + (kk >> 6) * WCHUNK + (kk & 7) * 2;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<unsigned short*>(
            chunk + sw128_offset((uint32_t)(half * 8 + q), (uint32_t)((kk & 63) >> 3))) = e[q];
    }
  });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    if (lane == 0) {
      // the recurrent product is needed for every step except the last one processed
      for (int step = 0; step + 1 < T; ++step) {
        grid_wait(ctr, (unsigned int)nC * (step + 1));   // dgh of this step is complete
        GRU_STAMP(0);
        tma_gather(s, tm, (step & 1) * Bp, Bp, nchunks, p.ring, p.gc, step, crank, csize);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step) {
        mma_consume<16>(s, tmem_base, nchunks, WCHUNK, Bp, p.ring, p.gc, step, csize);
        GRU_STAMP(2);
      }
    }
  } else {
    const int row = (warp & 3) * 32 + lane;
    const int uh = warp >> 2;
    const int ju = j0 + uh * GRU_UPT;
    const bool active = row < Bp;
    float dh_rec[GRU_UPT];   // dL/dh_t arriving through the recurrence (own units)
    GruGrad<GRU_UPT> db;
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      dh_rec[jj] = 0.f; db.r[jj] = 0.f; db.z[jj] = 0.f; db.n[jj] = 0.f; db.nr[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      // forward order of dir 0 is t=0..T-1, so its backward order is T-1..0; dir 1 mirrored
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;       // time index of h_{prev} in forward order
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + row;
      GruGates<GRU_UPT> a;
      float dh[GRU_UPT], hp[GRU_UPT];
      if (active) gru_load_bwd(p, m, (long long)tp * Bp + row, has_prev, dir, ju, a, dh, hp);
      // ---- recurrent part of dL/dh_t: product issued in the previous step ----
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        uint32_t v[8];
        tmem_ld_32x32b_x8(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + uh * GRU_UPT, v);
        tmem_ld_wait();
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) dh_rec[jj] += __uint_as_float(v[jj]);
      }
      GruGrad<GRU_UPT> d;
      if (active) gru_cell_bwd(a, dh, hp, dh_rec, d, db);
      gru_publish_bwd(p, step, tid, active, xb + (long long)row * K3 + ju, d, ctr);
      if (active) gru_store_bwd(p, m, dir, ju, d);
      if (tid == 0) GRU_STAMP(10);
    }
    // ---- bias gradients: reduce the per-batch-row partial sums over the CTA ----
    epi_barrier();
    float* red = s.scratch;  // [64]: r(16) z(16) n(16) hn(16)
    if (tid < 64) red[tid] = 0.f;
    epi_barrier();
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      const float a = warp_sum(active ? db.r[jj] : 0.f);
      const float b = warp_sum(active ? db.z[jj] : 0.f);
      const float c = warp_sum(active ? db.n[jj] : 0.f);
      const float d = warp_sum(active ? db.nr[jj] : 0.f);
      if (lane == 0) {
        atomicAdd(&red[uh * GRU_UPT + jj], a);
        atomicAdd(&red[16 + uh * GRU_UPT + jj], b);
        atomicAdd(&red[32 + uh * GRU_UPT + jj], c);
        atomicAdd(&red[48 + uh * GRU_UPT + jj], d);
      }
    }
    epi_barrier();
    if (tid < 48) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      const int idx = dir * K3 + g * H + j0 + jj;
      atomicAdd(p.dbih + idx, red[tid]);
      atomicAdd(p.dbhh + idx, g < 2 ? red[tid] : red[48 + jj]);
    }
  }
  gru_teardown(tmem_base, 32);
}

// =============================================================================================
// backward, K-split variant: the 4 CTAs of a cluster jointly own 64 hidden units.
//
// The plain backward kernel makes every CTA gather ALL of dgh_t (Bp x 3H bf16 = 384 KB at the
// north-star size) every step; with 96 KB of weights resident only 128 KB can be in flight, so
// the gather alone costs ~9 us of the 15.8 us step.  Here CTA r of a cluster contracts only the
// r-th QUARTER of the K = 3H dimension, for all 64 units of its cluster:
//     D_r[batch x 64] = dgh_t[:, quarter r] * W_hh[quarter r, 64 units]          (96 KB gathered)
// and the four partial products are reduce-scattered through distributed shared memory: for each
// peer in turn, the epilogue stages the 16 columns that belong to it in local shared memory and
// sends them with ONE bulk copy into the peer's receive buffer, completing on the peer's mbarrier;
// the owner adds the three slices it received to its own.  12 KB of DSMEM traffic replaces 288 KB
// of L2 reads per CTA per step.
// Requires cluster size 4, H % 256 == 0.
// =============================================================================================
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_bwd_ks_kernel(const __grid_constant__ CUtensorMap tm_d0,
                  const __grid_constant__ CUtensorMap tm_d1, const GruBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int cta_in_dir = blockIdx.x % nC;
  const int j0 = cta_in_dir * GRU_HC;                 // own 16 units (elementwise work)
  const uint32_t crank = cluster_rank();              // == cta_in_dir % 4
  const int k0c = (cta_in_dir / KS) * (KS * GRU_HC);  // first of the cluster's 64 units
  const int K3 = 3 * H;
  const int KQ = K3 / KS;                             // this CTA's share of the contraction
  const int nchunks = KQ / 64;
  const int stride = Bp * 128;
  const GruSmemLayout L = gru_layout_bwd_ks(Bp, H);
  const GruSmem s = gru_carve(smem_raw, L);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const int gc = gru_group_chunks(nchunks);
  const int ngroups = nchunks / gc;                   // <= GRU_KS_BWD_GROUPS: checked on the host

  const uint32_t tmem_base =
      gru_setup(s, L, tm, 64, KS, [&] { ks_stage_whh_t(s.wtile, p.whh, H, dir, k0c, crank); });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step) {
        grid_wait(ctr, (unsigned int)nC * (step + 1));   // dgh of this step is complete
        ks_gather_bwd(s, tm, stride, ngroups, gc, (int)crank * KQ, (step & 1) * Bp);
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step)
        ks_mma_bwd(s, tmem_base, stride, ngroups, gc, 64 * 128, umma_idesc_bf16_f32(128, 64),
                   false, step & 1);
    }
  } else {
    const int row = (warp & 3) * 32 + lane;
    const int uh = warp >> 2;
    const int ju = j0 + uh * GRU_UPT;
    const bool active = row < Bp;
    float dh_rec[GRU_UPT];
    GruGrad<GRU_UPT> db;
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      dh_rec[jj] = 0.f; db.r[jj] = 0.f; db.z[jj] = 0.f; db.n[jj] = 0.f; db.nr[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + row;
      GruGates<GRU_UPT> a;
      float dh[GRU_UPT], hp[GRU_UPT];
      if (active) gru_load_bwd(p, m, (long long)tp * Bp + row, has_prev, dir, ju, a, dh, hp);
      // ---- recurrent part of dL/dh_t: reduce-scatter of the four partial products ----
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        float own[GRU_UPT];
        if (tid == 0) mbar_expect_tx(s.recvbar, (uint32_t)((KS - 1) * Bp * 16 * 4));
        // the peers' slices first, each staged and sent as soon as it is complete (see
        // gru_fwd_ks_kernel); the own slice last
#pragma unroll 1
        for (int q = 1; q <= KS; ++q) {
          const uint32_t pr = (crank + (uint32_t)q) % KS;      // q == KS: own slice
          uint32_t v[8];
          tmem_ld_32x32b_x8(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + pr * 16 +
                                uh * GRU_UPT, v);
          tmem_ld_wait();
          if (q == KS) {
#pragma unroll
            for (int jj = 0; jj < GRU_UPT; ++jj) own[jj] = __uint_as_float(v[jj]);
          } else {
            if (active) {
              float4* sp = reinterpret_cast<float4*>(s.stage + ((size_t)pr * Bp + row) * 16 +
                                                     uh * GRU_UPT);
              sp[0] = make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]),
                                  __uint_as_float(v[2]), __uint_as_float(v[3]));
              sp[1] = make_float4(__uint_as_float(v[4]), __uint_as_float(v[5]),
                                  __uint_as_float(v[6]), __uint_as_float(v[7]));
            }
            fence_proxy_async_smem();
            epi_barrier();
            if (tid == 0)
              bulk_s2peer(mapa_shared(smem_u32(s.recv + (size_t)crank * Bp * 16), pr),
                          s.stage + (size_t)pr * Bp * 16, (uint32_t)(Bp * 16 * 4),
                          mapa_shared(smem_u32(s.recvbar), pr));
          }
        }
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(s.recvbar, (step - 1) & 1);
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) dh_rec[jj] += own[jj];
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            if ((uint32_t)src == crank) continue;
            const float4* rp = reinterpret_cast<const float4*>(
                s.recv + ((size_t)src * Bp + row) * 16 + uh * GRU_UPT);
            const float4 a = rp[0], b = rp[1];
            dh_rec[0] += a.x; dh_rec[1] += a.y; dh_rec[2] += a.z; dh_rec[3] += a.w;
            dh_rec[4] += b.x; dh_rec[5] += b.y; dh_rec[6] += b.z; dh_rec[7] += b.w;
          }
        }
      }
      GruGrad<GRU_UPT> d;
      if (active) gru_cell_bwd(a, dh, hp, dh_rec, d, db);
      gru_publish_bwd(p, step, tid, active, xb + (long long)row * K3 + ju, d, ctr);
      if (active) gru_store_bwd(p, m, dir, ju, d);
      if (tid == 0) GRU_STAMP(10);
    }
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      const float a = warp_sum(active ? db.r[jj] : 0.f);
      const float b = warp_sum(active ? db.z[jj] : 0.f);
      const float c = warp_sum(active ? db.n[jj] : 0.f);
      const float d = warp_sum(active ? db.nr[jj] : 0.f);
      if (lane == 0) {
        const int bi = dir * K3 + ju + jj;
        atomicAdd(p.dbih + bi, a);
        atomicAdd(p.dbih + bi + H, b);
        atomicAdd(p.dbih + bi + 2 * H, c);
        atomicAdd(p.dbhh + bi, a);
        atomicAdd(p.dbhh + bi + H, b);
        atomicAdd(p.dbhh + bi + 2 * H, d);
      }
    }
  }
  gru_teardown(tmem_base, 64);
}

// =============================================================================================
// forward, K-split variant: the 4 CTAs of a cluster jointly own 64 hidden units.
//
// Measured on gru_fwd_kernel (globaltimer timeline, H = 1024, B = 64, 7.4 us/step): 3.5 us pass
// between "h_{t-1} is complete" and "all MMAs retired", for a gather of 128 KB per CTA - the same
// ~30 B/ns per SM whether it is fetched as tensor boxes or as contiguous bulk copies, with or
// without cluster multicast: 128 CTAs x 128 KB = 16 MB of L2->SM traffic per step is the bound,
// next to 480 KB of shared-memory traffic (TMA writes + MMA operand reads of a 128-row A tile).
// Here CTA r of a cluster contracts only the r-th QUARTER of K = H for all 64 units of its
// cluster and all three gates,
//     D_r[batch x 192] = h_{t-1}[:, quarter r] * W_hh[(r|z|n) x 64 units, quarter r]^T,
// i.e. it gathers 32 KB instead of 128 KB (the whole quarter stays resident: no ring) and issues
// 16 MMAs of N = 192 instead of 64 of N = 48; the four partial products are reduce-scattered
// through distributed shared memory exactly as in gru_bwd_ks_kernel (each CTA receives the
// 3 x 16 columns of its own units from its three peers: 36 KB per CTA and step).
// Requires cluster size 4, H % 256 == 0, Bp <= 64.
// =============================================================================================
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_fwd_ks_kernel(const __grid_constant__ CUtensorMap tm_d0,
                  const __grid_constant__ CUtensorMap tm_d1, const GruFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int cta_in_dir = blockIdx.x % nC;
  const int j0 = cta_in_dir * GRU_HC;                 // own 16 units (gate math, stores)
  const uint32_t crank = cluster_rank();              // == cta_in_dir % 4
  const int k0c = (cta_in_dir / KS) * (KS * GRU_HC);  // first of the cluster's 64 units
  const int KQ = H / KS;                              // this CTA's share of the contraction
  const int nchunks = KQ / 64;
  constexpr int NCOL = 3 * KS * GRU_HC;               // 192 accumulator columns: gate x 64 units
  constexpr int WCHUNK = NCOL * 128;                  // 192 rows x 64 bf16
  constexpr int RW = 3 * GRU_HC;                      // 48 floats received per row and peer
  const int stride = Bp * 128;
  const GruSmemLayout L = gru_layout_fwd_ks(Bp, H);
  const GruSmem s = gru_carve(smem_raw, L);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;

  const uint32_t tmem_base = gru_setup(s, L, tm, 256, KS, [&] {
    // resident operand: rows = (gate, unit of the cluster), columns = this CTA's K quarter
    const int pieces_per_row = nchunks * 8;
    for (int k = tid; k < NCOL * pieces_per_row; k += GRU_THREADS) {
      const int r = k / pieces_per_row, pc = k % pieces_per_row;
      const int g = r / (KS * GRU_HC), u = r % (KS * GRU_HC);
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * 3 * H + (long long)g * H + k0c + u) * H + (long long)crank * KQ +
          pc * 8);
      *reinterpret_cast<uint4*>(s.wtile + (pc >> 3) * WCHUNK + sw128_offset(r, pc & 7)) = v;
    }
    if (tid < RW) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      s.scratch[tid] = p.bhh[dir * 3 * H + g * H + j0 + jj];
    }
  });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    // ===================== TMA producer: this CTA's K quarter of h_{t-1} =====================
    if (lane == 0) {
      for (int step = 1; step < T; ++step) {
        const int t = dir == 0 ? step : (T - 1 - step);
        const int tp = dir == 0 ? t - 1 : t + 1;
        grid_wait(ctr, (unsigned int)nC * step);   // all CTAs published h_{tp}
        GRU_STAMP(0);
        if (p.dbg && step == 21) p.dbg[1024 + 256 + blockIdx.x] = gtime();   // skew probe
        ks_gather_fwd(s, tm, stride, nchunks, (int)crank * KQ, tp * Bp);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(128, NCOL);
      for (int step = 1; step < T; ++step) {
        ks_mma_fwd(s, tmem_base, stride, nchunks, WCHUNK, idesc, false, (step - 1) & 1);
        GRU_STAMP(2);
      }
    }
  } else {
    // ===================== epilogue: thread = (batch row, half of the CTA's 16 units) ==========
    const int row = (warp & 3) * 32 + lane;
    const int uh = warp >> 2;
    const int ju = j0 + uh * GRU_UPT;
    const bool active = row < Bp;
    float hprev[GRU_UPT];
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) hprev[jj] = 0.f;
    float bias[3][GRU_UPT];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int jj = 0; jj < GRU_UPT; ++jj) bias[g][jj] = s.scratch[g * GRU_HC + uh * GRU_UPT + jj];

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? step : (T - 1 - step);
      float gi[3][GRU_UPT];
      if (active) gru_load_gi(p, t, row, dir, ju, gi);
      float acc[3][GRU_UPT];
#pragma unroll
      for (int gg = 0; gg < 3; ++gg)
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) acc[gg][jj] = 0.f;
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        // ---- reduce-scatter of the four partial products.  The three slices that belong to
        // the peers go first, one at a time: TMEM -> registers -> local staging -> (named barrier)
        // -> ONE bulk copy into the peer's receive buffer, so the first copy is in flight while
        // the next slice is still being staged; the CTA's own slice is read last ----
        if (tid == 0) mbar_expect_tx(s.recvbar, (uint32_t)((KS - 1) * Bp * RW * 4));
#pragma unroll 1
        for (int q = 1; q <= KS; ++q) {
          const uint32_t pr = (crank + (uint32_t)q) % KS;      // q == KS: own slice
          uint32_t v[3][8];
#pragma unroll
          for (int gg = 0; gg < 3; ++gg)
            tmem_ld_32x32b_x8(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) +
                                  gg * (KS * GRU_HC) + pr * GRU_HC + uh * GRU_UPT, v[gg]);
          tmem_ld_wait();
          if (q == KS) {
#pragma unroll
            for (int gg = 0; gg < 3; ++gg)
#pragma unroll
              for (int jj = 0; jj < GRU_UPT; ++jj) acc[gg][jj] = __uint_as_float(v[gg][jj]);
          } else {
            if (active) {
              float* sp = s.stage + ((size_t)pr * Bp + row) * RW + uh * GRU_UPT;
#pragma unroll
              for (int gg = 0; gg < 3; ++gg) {
                float4* o = reinterpret_cast<float4*>(sp + gg * GRU_HC);
                o[0] = make_float4(__uint_as_float(v[gg][0]), __uint_as_float(v[gg][1]),
                                   __uint_as_float(v[gg][2]), __uint_as_float(v[gg][3]));
                o[1] = make_float4(__uint_as_float(v[gg][4]), __uint_as_float(v[gg][5]),
                                   __uint_as_float(v[gg][6]), __uint_as_float(v[gg][7]));
              }
            }
            fence_proxy_async_smem();   // generic st.shared -> the copy engine's (async proxy) reads
            epi_barrier();              // this peer's slice is completely staged
            if (tid == 0)
              bulk_s2peer(mapa_shared(smem_u32(s.recv + (size_t)crank * Bp * RW), pr),
                          s.stage + (size_t)pr * Bp * RW, (uint32_t)(Bp * RW * 4),
                          mapa_shared(smem_u32(s.recvbar), pr));
          }
        }
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(s.recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            if ((uint32_t)src == crank) continue;
            const float* rp = s.recv + ((size_t)src * Bp + row) * RW + uh * GRU_UPT;
#pragma unroll
            for (int gg = 0; gg < 3; ++gg) {
              const float4 a = *reinterpret_cast<const float4*>(rp + gg * GRU_HC);
              const float4 b = *reinterpret_cast<const float4*>(rp + gg * GRU_HC + 4);
              acc[gg][0] += a.x; acc[gg][1] += a.y; acc[gg][2] += a.z; acc[gg][3] += a.w;
              acc[gg][4] += b.x; acc[gg][5] += b.y; acc[gg][6] += b.z; acc[gg][7] += b.w;
            }
          }
        }
      }
      const long long m = (long long)t * Bp + row;
      GruGates<GRU_UPT> g;
      if (active) gru_cell_fwd(gi, acc, bias, hprev, g);
      gru_publish_fwd(p, step, tid, active, p.xn + m * D + dir * H + ju, hprev, ctr, true);
      if (active) gru_store_fwd(p, m, dir, ju, hprev, g);
      if (tid == 0) GRU_STAMP(10);
    }
  }
  gru_teardown(tmem_base, 256);
}

// =============================================================================================
// forward, K split with the accumulator TRANSPOSED: D^T[(gate, unit) x batch].
//
// Same partition as gru_fwd_ks_kernel (cluster of 4 owns 64 units, CTA r contracts K quarter r),
// but the resident weight slice is the M-side operand and h_{t-1} the N-side one:
//     D0[128 x Bp] = W[(r|z) x 64 units, quarter r] * h_{t-1}[:, quarter r]^T     (TMEM cols 0..)
//     D1[ 64 x Bp] = W[ n    x 64 units, quarter r] * h_{t-1}[:, quarter r]^T     (TMEM cols 64..)
// An MMA of N = Bp costs Bp/256 of the N = 192 one, so the tensor-core share of the step falls
// from 16 x 96 to 32 x (Bp/8) cycles (1536 -> 1024 at 64 rows, -> 128 at 8 rows), and every
// accumulator lane is a weight row, so all 128 lanes (all four TMEM sub-partitions) carry data
// whatever the batch is.  The weight rows are ordered by OWNER: tile 0 rows 32q..32q+31 are the
// r and z rows of the 16 units CTA q of the cluster owns, tile 1 rows 16q..16q+15 its n rows, so
// an epilogue thread's accumulator row goes to exactly one peer: it is written as one row of
// [48][Bp] (pitch Bp+4: conflict-free) into the staging slice for that peer, the three slices leave
// as one bulk copy each, and the gate math then runs on ALL 256 epilogue threads
// (thread = batch row x UPT units) from the four received slices.
// Requires cluster size 4, H % 256 == 0, Bp <= 64 (Bp % 8 == 0 as everywhere).
// =============================================================================================
template <int UPT>
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_fwd_kt_kernel(const __grid_constant__ CUtensorMap tm_d0,
                  const __grid_constant__ CUtensorMap tm_d1, const GruFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int cta_in_dir = blockIdx.x % nC;
  const int j0 = cta_in_dir * GRU_HC;                 // own 16 units (gate math, stores)
  const uint32_t crank = cluster_rank();              // == cta_in_dir % 4
  const int k0c = (cta_in_dir / KS) * (KS * GRU_HC);  // first of the cluster's 64 units
  const int KQ = H / KS;                              // this CTA's share of the contraction
  const int nchunks = KQ / 64;
  constexpr int WROWS = 3 * KS * GRU_HC;              // 192 weight rows: 128 (r,z) + 64 (n)
  constexpr int WCHUNK = WROWS * 128;                 // 192 rows x 64 bf16
  constexpr int RW = 3 * GRU_HC;                      // 48 accumulator rows per owner
  const int P = Bp + 4;                               // pitch of a staged row (floats)
  const int slice = RW * P;                           // floats per (source, owner) slice
  const int NB = (Bp + 15) & ~15;                     // MMA N (rows of h read per chunk)
  const int stride = Bp * 128;
  const GruSmemLayout L = gru_layout_fwd_kt(Bp, H);
  const GruSmem s = gru_carve(smem_raw, L);           // recv [KS src][48][P], stage [KS-1 dst]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;

  const uint32_t tmem_base = gru_setup(s, L, tm, 128, KS, [&] {
    // resident operand: rows ordered by owner (see above), columns = this CTA's K quarter
    const int pieces_per_row = nchunks * 8;
    for (int k = tid; k < WROWS * pieces_per_row; k += GRU_THREADS) {
      const int r = k / pieces_per_row, pc = k % pieces_per_row;
      int g, u;
      if (r < 128) { g = (r & 31) >> 4; u = (r >> 5) * GRU_HC + (r & 15); }
      else { g = 2; u = r - 128; }
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * 3 * H + (long long)g * H + k0c + u) * H + (long long)crank * KQ +
          pc * 8);
      *reinterpret_cast<uint4*>(s.wtile + (pc >> 3) * WCHUNK + sw128_offset(r, pc & 7)) = v;
    }
    if (tid < RW) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      s.scratch[tid] = p.bhh[dir * 3 * H + g * H + j0 + jj];
    }
  });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    // ===================== TMA producer: this CTA's K quarter of h_{t-1} =====================
    if (lane == 0) {
      for (int step = 1; step < T; ++step) {
        const int t = dir == 0 ? step : (T - 1 - step);
        const int tp = dir == 0 ? t - 1 : t + 1;
        grid_wait(ctr, (unsigned int)nC * step);   // all CTAs published h_{tp}
        GRU_STAMP(0);
        if (p.dbg && step == 21) p.dbg[1024 + 256 + blockIdx.x] = gtime();   // skew probe
        ks_gather_fwd(s, tm, stride, nchunks, (int)crank * KQ, tp * Bp);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(128, (uint32_t)NB);
      for (int step = 1; step < T; ++step) {
        ks_mma_fwd(s, tmem_base, stride, nchunks, WCHUNK, idesc, true, (step - 1) & 1);
        GRU_STAMP(2);
      }
    }
  } else {
    // ===================== epilogue =====================
    // phase A (scatter): warp w reads accumulator lanes 32*(w&3).. of tile 0 and, for w&3 < 2,
    // of tile 1, for the column blocks (8 batch rows each) of its half (w>>2) of the batch
    const int sub = warp & 3, hi = warp >> 2;
    const int nblk = Bp >> 3;
    const int blk0 = hi == 0 ? 0 : (nblk + 1) / 2;
    const int myblk = hi == 0 ? (nblk + 1) / 2 : nblk / 2;          // <= 4
    const uint32_t own0 = (uint32_t)sub;                            // owner of the tile-0 row
    const uint32_t own1 = (uint32_t)(sub * 2 + (lane >> 4));        // owner of the tile-1 row
    const uint32_t q0 = (own0 + KS - crank) % KS, q1 = (own1 + KS - crank) % KS;
    float* dst0 = (q0 == 0 ? s.recv + crank * slice : s.stage + (q0 - 1) * slice) + lane * P;
    float* dst1 = (q1 == 0 ? s.recv + crank * slice : s.stage + (q1 - 1) * slice) +
                  (2 * GRU_HC + (lane & 15)) * P;
    // phase B (gate math): thread = (batch row b, UPT of the CTA's 16 units)
    const int b = tid % Bp, ug = tid / Bp;
    const bool active = ug * UPT < GRU_HC;
    const int u0 = ug * UPT;
    const int ju = j0 + u0;
    float hprev[UPT];
#pragma unroll
    for (int jj = 0; jj < UPT; ++jj) hprev[jj] = 0.f;
    float bias[3][UPT];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int jj = 0; jj < UPT; ++jj) bias[g][jj] = active ? s.scratch[g * GRU_HC + u0 + jj] : 0.f;

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? step : (T - 1 - step);
      float gi[3][UPT];
      if (active) gru_load_gi(p, t, b, dir, ju, gi);
      float acc[3][UPT];
#pragma unroll
      for (int gg = 0; gg < 3; ++gg)
#pragma unroll
        for (int jj = 0; jj < UPT; ++jj) acc[gg][jj] = 0.f;
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        if (tid == 0) mbar_expect_tx(s.recvbar, (uint32_t)((KS - 1) * slice * 4));
        {
          const uint32_t tl = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(blk0 * 8);
#pragma unroll
          for (int kb = 0; kb < 4; kb += 2) {
            if (kb < myblk) {
              uint32_t v0[2][8], v1[2][8];
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                if (kb + k < myblk) {
                  tmem_ld_32x32b_x8(tl + (kb + k) * 8, v0[k]);
                  if (sub < 2) tmem_ld_32x32b_x8(tl + 64 + (kb + k) * 8, v1[k]);
                }
              }
              tmem_ld_wait();
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                if (kb + k < myblk) {
                  float4* o = reinterpret_cast<float4*>(dst0 + (blk0 + kb + k) * 8);
                  o[0] = make_float4(__uint_as_float(v0[k][0]), __uint_as_float(v0[k][1]),
                                     __uint_as_float(v0[k][2]), __uint_as_float(v0[k][3]));
                  o[1] = make_float4(__uint_as_float(v0[k][4]), __uint_as_float(v0[k][5]),
                                     __uint_as_float(v0[k][6]), __uint_as_float(v0[k][7]));
                  if (sub < 2) {
                    float4* o1 = reinterpret_cast<float4*>(dst1 + (blk0 + kb + k) * 8);
                    o1[0] = make_float4(__uint_as_float(v1[k][0]), __uint_as_float(v1[k][1]),
                                        __uint_as_float(v1[k][2]), __uint_as_float(v1[k][3]));
                    o1[1] = make_float4(__uint_as_float(v1[k][4]), __uint_as_float(v1[k][5]),
                                        __uint_as_float(v1[k][6]), __uint_as_float(v1[k][7]));
                  }
                }
              }
            }
          }
        }
        tc_fence_before_sync();
        fence_proxy_async_smem();   // generic st.shared -> the copy engine's (async proxy) reads
        epi_barrier();              // all three outgoing slices (and the own one) are staged
        if (lane == 0 && warp >= 1 && warp <= KS - 1) {
          const uint32_t pr = (crank + (uint32_t)warp) % KS;
          bulk_s2peer(mapa_shared(smem_u32(s.recv + (size_t)crank * slice), pr),
                      s.stage + (size_t)(warp - 1) * slice, (uint32_t)(slice * 4),
                      mapa_shared(smem_u32(s.recvbar), pr));
        }
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(s.recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            const float* rp = s.recv + (size_t)src * slice + u0 * P + b;
#pragma unroll
            for (int gg = 0; gg < 3; ++gg)
#pragma unroll
              for (int jj = 0; jj < UPT; ++jj) acc[gg][jj] += rp[(gg * GRU_HC + jj) * P];
          }
        }
      }
      const long long m = (long long)t * Bp + b;
      GruGates<UPT> g;
      if (active) gru_cell_fwd(gi, acc, bias, hprev, g);
      gru_publish_fwd(p, step, tid, active, p.xn + m * D + dir * H + ju, hprev, ctr, true);
      if (active) gru_store_fwd(p, m, dir, ju, hprev, g);
      if (tid == 0) GRU_STAMP(10);
    }
  }
  gru_teardown(tmem_base, 128);
}

// =============================================================================================
// backward, K split with the accumulator TRANSPOSED (see gru_fwd_kt_kernel):
//     D^T[64 units x Bp] = W_hh^T[64 units of the cluster, quarter r of 3H] * dgh[:, quarter r]^T
// The weight tile is the one of gru_bwd_ks_kernel (its 64 rows are already grouped by owner);
// an accumulator lane is a unit, so its row of Bp partial sums goes to exactly one peer, and the
// elementwise work runs on all 256 epilogue threads (thread = batch row x 1 unit; the 128-row
// M-side read covers the next weight chunk with its lanes 64..127, which are never read).
// =============================================================================================
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_bwd_kt_kernel(const __grid_constant__ CUtensorMap tm_d0,
                  const __grid_constant__ CUtensorMap tm_d1, const GruBwdParams p) {
  constexpr int UPT = 1;
  extern __shared__ uint8_t smem_raw[];
  const int H = p.H, Bp = p.Bp, T = p.T;
  const int nC = H / GRU_HC;
  const int dir = blockIdx.x / nC;
  const int cta_in_dir = blockIdx.x % nC;
  const int j0 = cta_in_dir * GRU_HC;                 // own 16 units (elementwise work)
  const uint32_t crank = cluster_rank();              // == cta_in_dir % 4
  const int k0c = (cta_in_dir / KS) * (KS * GRU_HC);  // first of the cluster's 64 units
  const int K3 = 3 * H;
  const int KQ = K3 / KS;                             // this CTA's share of the contraction
  const int nchunks = KQ / 64;
  const int P = Bp + 4;                               // pitch of a staged row (floats)
  const int slice = GRU_HC * P;                       // floats per (source, owner) slice
  const int NB = (Bp + 15) & ~15;
  const int stride = Bp * 128;
  const GruSmemLayout L = gru_layout_bwd_kt(Bp, H);
  const GruSmem s = gru_carve(smem_raw, L);           // recv [KS src][16][P], stage [KS-1 dst]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const int gc = gru_group_chunks(nchunks);
  const int ngroups = nchunks / gc;                   // <= GRU_KS_BWD_GROUPS: checked on the host

  const uint32_t tmem_base =
      gru_setup(s, L, tm, 64, KS, [&] { ks_stage_whh_t(s.wtile, p.whh, H, dir, k0c, crank); });
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step) {
        grid_wait(ctr, (unsigned int)nC * (step + 1));   // dgh of this step is complete
        GRU_STAMP(0);
        ks_gather_bwd(s, tm, stride, ngroups, gc, (int)crank * KQ, (step & 1) * Bp);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(128, (uint32_t)NB);
      for (int step = 0; step + 1 < T; ++step) {
        ks_mma_bwd(s, tmem_base, stride, ngroups, gc, 64 * 128, idesc, true, step & 1);
        GRU_STAMP(2);
      }
    }
  } else {
    // phase A (scatter): warps with (w&3) < 2 hold the 64 valid accumulator lanes
    const int sub = warp & 3, hi = warp >> 2;
    const int nblk = Bp >> 3;
    const int blk0 = hi == 0 ? 0 : (nblk + 1) / 2;
    const int myblk = hi == 0 ? (nblk + 1) / 2 : nblk / 2;          // <= 4
    const uint32_t own = (uint32_t)(sub * 2 + (lane >> 4));
    const uint32_t q0 = (own + KS - crank) % KS;
    float* dst0 =
        (q0 == 0 ? s.recv + crank * slice : s.stage + (q0 - 1) * slice) + (lane & 15) * P;
    // phase B: thread = (batch row b, one of the CTA's 16 units)
    const int b = tid % Bp, ug = tid / Bp;
    const bool active = ug * UPT < GRU_HC;
    const int u0 = ug * UPT;
    const int ju = j0 + u0;
    float dh_rec[UPT];
    GruGrad<UPT> db;
#pragma unroll
    for (int jj = 0; jj < UPT; ++jj) {
      dh_rec[jj] = 0.f; db.r[jj] = 0.f; db.z[jj] = 0.f; db.n[jj] = 0.f; db.nr[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + b;
      GruGates<UPT> a;
      float dh[UPT], hp[UPT];
      if (active) gru_load_bwd(p, m, (long long)tp * Bp + b, has_prev, dir, ju, a, dh, hp);
      if (step > 0) {
        mbar_wait(s.accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        if (tid == 0) mbar_expect_tx(s.recvbar, (uint32_t)((KS - 1) * slice * 4));
        if (sub < 2) {
          const uint32_t tl = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(blk0 * 8);
          uint32_t v[4][8];
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < myblk) tmem_ld_32x32b_x8(tl + k * 8, v[k]);
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (k < myblk) {
              float4* o = reinterpret_cast<float4*>(dst0 + (blk0 + k) * 8);
              o[0] = make_float4(__uint_as_float(v[k][0]), __uint_as_float(v[k][1]),
                                 __uint_as_float(v[k][2]), __uint_as_float(v[k][3]));
              o[1] = make_float4(__uint_as_float(v[k][4]), __uint_as_float(v[k][5]),
                                 __uint_as_float(v[k][6]), __uint_as_float(v[k][7]));
            }
          }
        }
        tc_fence_before_sync();
        fence_proxy_async_smem();
        epi_barrier();
        if (lane == 0 && warp >= 1 && warp <= KS - 1) {
          const uint32_t pr = (crank + (uint32_t)warp) % KS;
          bulk_s2peer(mapa_shared(smem_u32(s.recv + (size_t)crank * slice), pr),
                      s.stage + (size_t)(warp - 1) * slice, (uint32_t)(slice * 4),
                      mapa_shared(smem_u32(s.recvbar), pr));
        }
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(s.recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            const float* rp = s.recv + (size_t)src * slice + u0 * P + b;
#pragma unroll
            for (int jj = 0; jj < UPT; ++jj) dh_rec[jj] += rp[jj * P];
          }
        }
      }
      GruGrad<UPT> d;
      if (active) gru_cell_bwd(a, dh, hp, dh_rec, d, db);
      gru_publish_bwd(p, step, tid, active, xb + (long long)b * K3 + ju, d, ctr);
      if (active) gru_store_bwd(p, m, dir, ju, d);
      if (tid == 0) GRU_STAMP(10);
    }
    if (active) {
#pragma unroll
      for (int jj = 0; jj < UPT; ++jj) {
        const int bi = dir * K3 + ju + jj;
        atomicAdd(p.dbih + bi, db.r[jj]);
        atomicAdd(p.dbih + bi + H, db.z[jj]);
        atomicAdd(p.dbih + bi + 2 * H, db.n[jj]);
        atomicAdd(p.dbhh + bi, db.r[jj]);
        atomicAdd(p.dbhh + bi + H, db.z[jj]);
        atomicAdd(p.dbhh + bi + 2 * H, db.nr[jj]);
      }
    }
  }
  gru_teardown(tmem_base, 64);
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, long long rows, long long cols,
                      long long ld, int box_rows);

static constexpr int GRU_SMEM_MAX = 227 * 1024;   // dynamic shared memory of one sm_100 CTA

// chunks are grouped gc per mbarrier pair (gc = largest of 4,3,2,1 dividing nchunks, or 1 when
// that leaves no ring); ring = the largest divisor of ngroups (<= GRU_MAX_RING) whose slots fit
// next to the resident weights
static int gru_ring_slots(int Bp, int nchunks, int wrows, int* gc_out, size_t* smem_bytes) {
  const int fixed = gru_layout_full(Bp, nchunks, wrows, 0).bytes;
  for (int gc : {gru_group_chunks(nchunks), 1}) {
    const int ngroups = nchunks / gc;
    const int fit = std::min((GRU_SMEM_MAX - fixed) / (gc * Bp * 128), GRU_MAX_RING);
    for (int r = fit; r >= 1; --r) {
      if (ngroups % r == 0) {
        *gc_out = gc;
        *smem_bytes = (size_t)gru_layout_full(Bp, nchunks, wrows, r * gc * Bp * 128).bytes;
        return r;
      }
    }
  }
  return -1;
}

static int g_gru_last_cluster = 0;
static unsigned long long* g_gru_dbg = nullptr;

// Which K-split flavour: the transposed-accumulator kernels (gru_*_kt_kernel) win while the batch
// is small.  Measured us/step at H = 1024 (kt | ks): forward 3.8 | 4.8 at 8 rows, 4.3 | 4.9 at 16,
// 5.3 | 5.4 at 32, 7.9 | 7.1 at 64; backward 4.6 | 5.3 at 8, 5.4 | 5.4 at 16, 6.2 | 5.8 at 32,
// 8.3 | 7.8 at 64.
static bool gru_use_kt(int Bp, bool backward) { return Bp <= (backward ? 8 : 32); }

// Every GRU kernel synchronises each direction through a grid barrier in global memory, so the
// whole grid must be resident at once.  Launches are not flagged cooperative: co-residency is
// proven with the occupancy API (one CTA per SM, grid <= resident capacity), and every spin-wait
// in the kernels is bounded.  The cluster size starts at cs_pref and halves while it does not
// divide the nC CTAs of a direction or the grid does not fit, down to cs_min; SB_ERR_UNSUPPORTED
// when no size fits, so that the caller can fall back to another kernel.
static int gru_launch(const void* kernel, int grid, int nC, int cs_pref, int cs_min, size_t smem,
                      void** args, cudaStream_t stream) {
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
      cudaSuccess) {
    cudaGetLastError();
    return SB_ERR_CUDA;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GRU_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.y = 1;
  attr.val.clusterDim.z = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  for (int cs = cs_pref; cs >= cs_min; cs >>= 1) {
    if (nC % cs != 0) continue;
    attr.val.clusterDim.x = cs;
    int resident = 0;
    cudaError_t e;
    if (cs > 1) {
      e = cudaOccupancyMaxActiveClusters(&resident, kernel, &cfg);
      resident *= cs;
    } else {
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, GRU_THREADS, smem);
      resident *= device_sm_count();
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    if (resident < grid) continue;
    if (cudaLaunchKernelExC(&cfg, kernel, args) != cudaSuccess) {
      cudaGetLastError();
      return SB_ERR_CUDA;
    }
    g_gru_last_cluster = cs;
    return SB_OK;
  }
  return SB_ERR_UNSUPPORTED;
}

// The tensor maps of the gathered operand, one per direction (direction 1 aliases direction 0
// when the layer is unidirectional): `rows` x `cols` bf16 with leading dimension `ld`, the
// direction's block starting `dir_stride` elements after the previous one, boxes of Bp rows.
static int gru_tmaps(CUtensorMap (&tm)[2], const bf16* base, long long rows, long long cols,
                     long long ld, size_t dir_stride, int ndir, int Bp) {
  for (int d = 0; d < 2; ++d) {
    const int rc = make_tmap_bf16_2d(&tm[d], base + (d < ndir ? d : 0) * dir_stride, rows, cols,
                                     ld, Bp);
    if (rc != SB_OK) return rc;
  }
  return SB_OK;
}

// workspace of one recurrence launch: [0,1024) the per-direction grid-barrier words, then the
// exchange buffers of the backward kernels
static constexpr size_t GRU_WS_COUNTERS = 1024;

}  // namespace sb

using namespace sb;

// developer hooks (not part of the drop-in surface)
extern "C" int sb_debug_gru_timeline(void* dev_buffer) {
  sb::g_gru_dbg = reinterpret_cast<unsigned long long*>(dev_buffer);
  return SB_OK;
}
extern "C" int sb_debug_gru_cluster(int query) {
  return query == 0 ? sb::g_gru_last_cluster : -1;
}

static int gru_check(int T, int Bp, int H, int ndir) {
  if (T <= 0 || Bp <= 0 || H <= 0 || (ndir != 1 && ndir != 2)) return SB_ERR_INVALID;
  if (H % GRU_HC != 0 || Bp % 8 != 0 || Bp > 128) return SB_ERR_UNSUPPORTED;
  if (ndir * (H / GRU_HC) > sb::device_sm_count()) return SB_ERR_UNSUPPORTED;
  return SB_OK;
}

// Common to sb_gru_fwd and sb_gru_bwd: validate the shape and the arguments, check the workspace
// (`need` bytes, 1024-aligned) and zero it: the grid-barrier counters start at 0, and so do the
// exchange tiles (columns past 3H of a partial chunk are never written and must read as zero).
static int gru_begin(int T, int Bp, int H, int ndir, bool args_ok, void* workspace,
                     size_t workspace_bytes, size_t need, cudaStream_t stream) {
  const int rc = gru_check(T, Bp, H, ndir);
  if (rc != SB_OK) return rc;
  if (!args_ok || !workspace) return SB_ERR_INVALID;
  if (workspace_bytes < need) return SB_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return SB_ERR_INVALID;
  if (cudaMemsetAsync(workspace, 0, need, stream) != cudaSuccess) return SB_ERR_CUDA;
  return SB_OK;
}

extern "C" int sb_gru_fwd_workspace_size(int Bp, int H, int ndir, size_t* bytes) {
  if (!bytes || Bp <= 0 || H <= 0 || (ndir != 1 && ndir != 2)) return SB_ERR_INVALID;
  (void)Bp;
  *bytes = GRU_WS_COUNTERS;      // the forward kernels exchange h_t through xn itself
  return SB_OK;
}

// Forward kernel selection: the K split over 4-CTA clusters (H % 256 == 0, batch rows <= 64) when
// its layout fits, kt rather than ks when gru_use_kt picks it and kt fits too; otherwise, or when a
// K-split grid cannot be co-resident, every CTA gathers all of h_{t-1} (TMA, cluster multicast).
static int gru_fwd_select(GruFwdParams& p, void** args, cudaStream_t stream) {
  const int H = p.H, Bp = p.Bp, grid = p.ndir * (H / GRU_HC), nC = H / GRU_HC;
  int gc = 1;
  size_t smem = 0;
  const int ring = gru_ring_slots(Bp, (H + 63) / 64, 48, &gc, &smem);
  if (ring < 0) return SB_ERR_UNSUPPORTED;
  if (H % 256 == 0 && Bp <= 64) {
    const GruSmemLayout ks = gru_layout_fwd_ks(Bp, H), kt = gru_layout_fwd_kt(Bp, H);
    if (ks.bytes <= GRU_SMEM_MAX) {
      p.ring = H / KS / 64;
      p.gc = 1;
      if (gru_use_kt(Bp, false) && kt.bytes <= GRU_SMEM_MAX) {
        const void* k = Bp > 16 ? (const void*)gru_fwd_kt_kernel<2> : (const void*)gru_fwd_kt_kernel<1>;
        if (gru_launch(k, grid, nC, KS, KS, kt.bytes, args, stream) == SB_OK) return SB_OK;
      }
      if (gru_launch((const void*)gru_fwd_ks_kernel, grid, nC, KS, KS, ks.bytes, args, stream) ==
          SB_OK)
        return SB_OK;
    }
  }
  p.ring = ring;
  p.gc = gc;
  return gru_launch((const void*)gru_fwd_kernel, grid, nC, 4, 1, smem, args, stream);
}

extern "C" int sb_gru_fwd(const float* gi, const void* whh_bf16, const float* bhh, float* y,
                          void* xn_bf16, float* gates, void* workspace, size_t workspace_bytes,
                          int T, int Bp, int H, int ndir, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  size_t need = 0;
  sb_gru_fwd_workspace_size(Bp, H, ndir, &need);
  int rc = gru_begin(T, Bp, H, ndir, gi && whh_bf16 && bhh && y && xn_bf16, workspace,
                     workspace_bytes, need, stream);
  if (rc != SB_OK) return rc;
  GruFwdParams p;
  p.gi = gi; p.whh = reinterpret_cast<const bf16*>(whh_bf16); p.bhh = bhh; p.y = y;
  p.xn = reinterpret_cast<bf16*>(xn_bf16);
  p.gates = gates; p.barrier = reinterpret_cast<unsigned int*>(workspace);
  p.T = T; p.Bp = Bp; p.H = H; p.ndir = ndir;
  p.dbg = g_gru_dbg;
  CUtensorMap tm[2];
  rc = gru_tmaps(tm, p.xn, (long long)T * Bp, H, (long long)ndir * H, (size_t)H, ndir, Bp);
  if (rc != SB_OK) return rc;
  void* args[] = {(void*)&tm[0], (void*)&tm[1], (void*)&p};
  return gru_fwd_select(p, args, stream);
}

extern "C" int sb_gru_bwd_workspace_size(int Bp, int H, int ndir, size_t* bytes) {
  if (!bytes || Bp <= 0 || H <= 0 || (ndir != 1 && ndir != 2)) return SB_ERR_INVALID;
  // counters + the double-buffered exchange of dgh_t (Bp x 3H bf16 per direction and parity; the
  // tile-major form of the K-split kernel rounds 3H up to whole 64-column chunks)
  const size_t k3p = (size_t)((3 * H + 63) / 64) * 64;
  *bytes = GRU_WS_COUNTERS + (size_t)ndir * 2 * Bp * k3p * sizeof(bf16) + 1024;
  return SB_OK;
}

// Backward kernel selection, the chain of the forward one: the K split when its chunk groups fit
// its full barriers and its layout fits (kt rather than ks when gru_use_kt picks it and kt fits
// too), otherwise the full gather.
static int gru_bwd_select(GruBwdParams& p, void** args, cudaStream_t stream) {
  const int H = p.H, Bp = p.Bp, grid = p.ndir * (H / GRU_HC), nC = H / GRU_HC;
  const int nchunks = (3 * H + 63) / 64;
  if (H % 256 == 0) {
    const GruSmemLayout ks = gru_layout_bwd_ks(Bp, H), kt = gru_layout_bwd_kt(Bp, H);
    const int nq = 3 * H / KS / 64;
    if (nq / gru_group_chunks(nq) <= ks.nfull && ks.bytes <= GRU_SMEM_MAX) {
      p.ring = nq;
      p.gc = 1;
      if (gru_use_kt(Bp, true) && kt.bytes <= GRU_SMEM_MAX &&
          gru_launch((const void*)gru_bwd_kt_kernel, grid, nC, KS, KS, kt.bytes, args, stream) ==
              SB_OK)
        return SB_OK;
      if (gru_launch((const void*)gru_bwd_ks_kernel, grid, nC, KS, KS, ks.bytes, args, stream) ==
          SB_OK)
        return SB_OK;
    }
  }
  size_t smem = 0;
  p.ring = gru_ring_slots(Bp, nchunks, 16, &p.gc, &smem);
  if (p.ring < 0) return SB_ERR_UNSUPPORTED;
  return gru_launch((const void*)gru_bwd_kernel, grid, nC, 4, 1, smem, args, stream);
}

extern "C" int sb_gru_bwd(const float* dy, const float* y, const float* gates,
                          const void* whh_bf16, void* dgi_bf16, void* dghn_bf16, float* dbih,
                          float* dbhh, void* workspace, size_t workspace_bytes, int T, int Bp,
                          int H, int ndir, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  size_t need = 0;
  sb_gru_bwd_workspace_size(Bp, H, ndir, &need);
  int rc = gru_begin(T, Bp, H, ndir,
                     dy && y && gates && whh_bf16 && dgi_bf16 && dghn_bf16 && dbih && dbhh,
                     workspace, workspace_bytes, need, stream);
  if (rc != SB_OK) return rc;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  GruBwdParams p;
  p.dy = dy; p.y = y; p.gates = gates; p.whh = reinterpret_cast<const bf16*>(whh_bf16);
  p.dgi = reinterpret_cast<bf16*>(dgi_bf16);
  p.dghn = reinterpret_cast<bf16*>(dghn_bf16);
  p.barrier = reinterpret_cast<unsigned int*>(ws);
  p.xchg = reinterpret_cast<bf16*>(ws + GRU_WS_COUNTERS);
  p.dbih = dbih; p.dbhh = dbhh; p.T = T; p.Bp = Bp; p.H = H; p.ndir = ndir;
  p.dbg = g_gru_dbg;
  // per direction: the two parity buffers stacked as [2*Bp rows][3H cols]
  const int K3 = 3 * H;
  CUtensorMap tm[2];
  rc = gru_tmaps(tm, p.xchg, 2LL * Bp, K3, K3, (size_t)2 * Bp * K3, ndir, Bp);
  if (rc != SB_OK) return rc;
  void* args[] = {(void*)&tm[0], (void*)&tm[1], (void*)&p};
  return gru_bwd_select(p, args, stream);
}
