// Persistent GRU recurrence kernels (forward and backward in time) for sm_100a.
//
// Replaces the cuDNN RNN reached through nn.GRU in the reference encoder
// (speech/models/model.py:35-39 construction, :73 call; gate order r,z,n; bidirectional halves
// are summed by the caller, model.py:75-77) and the pred-net GRU of the transducer
// (speech/models/transducer_model.py:23-26,68).
//
// The time-batched input projection gi = X W_ih^T + b_ih is done for all T at once by
// sb_gemm_bf16_tn; these kernels run the T-serial part.  One launch per layer covers BOTH
// directions:
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
//     barrier, and only then write the fp32 state / saved gates;
//   * the grid barrier is one red.release.gpu + ld.acquire.gpu polling on a global counter.
// The backward kernel has the same structure with W_hh^T resident (16 rows x 3H) and the
// all-gather over the pre-activation gradients dgh_t (batch x 3H).
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
static constexpr int GRU_UPT = 8;            // hidden units per epilogue thread
static constexpr int GRU_MAX_RING = 16;      // smem ring slots for the gathered operand
static constexpr int GRU_EPI = 256;          // warps 0..7: epilogue
static constexpr int GRU_THREADS = GRU_EPI + 64;  // + warp 8: MMA issuer/TMEM owner, warp 9: TMA

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

struct GruSmem {
  uint8_t* ring;    // ring slots (stride = Bp*128 bytes), placed BEFORE the weights so that the
                    // 128-row MMA read of the last slot overruns into (finite) weight data
  uint8_t* wtile;   // resident weight chunks
  uint64_t* full;   // [GRU_MAX_RING]
  uint64_t* empty;  // [GRU_MAX_RING]
  uint64_t* accfull;
  uint32_t* tmem_slot;
  float* scratch;   // [64]
};

SB_DEVINL GruSmem carve(uint8_t* raw, int ring_bytes, int wbytes) {
  GruSmem s;
  s.ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) &
                                      ~static_cast<uintptr_t>(1023));
  s.wtile = s.ring + ring_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s.wtile + wbytes);
  s.full = bars;
  s.empty = bars + GRU_MAX_RING;
  s.accfull = bars + 2 * GRU_MAX_RING;
  s.tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * GRU_MAX_RING + 1);
  s.scratch = reinterpret_cast<float*>(bars + 2 * GRU_MAX_RING + 2);
  return s;
}

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

SB_DEVINL float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
SB_DEVINL float fast_tanh(float x) {
  // 1 - 2/(exp(2x)+1), clamped so exp never overflows (__fdividef(2, inf) is not guaranteed 0)
  const float xc = fminf(fmaxf(x, -15.f), 15.f);
  return 1.0f - __fdividef(2.0f, __expf(2.0f * xc) + 1.0f);
}

// One-touch data (gi, saved gates, dy, fp32 state, GEMM operands written for later kernels) uses
// the streaming cache policy (.cs) so that it does not evict the latency-critical bf16 exchange
// buffers, which every CTA re-reads from L2 each step.
SB_DEVINL void ld8(const float* p, float (&v)[8]) {
  const float4 a = __ldcs(reinterpret_cast<const float4*>(p));
  const float4 b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
SB_DEVINL void st8(float* p, const float (&v)[8]) {
  __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  __stcs(reinterpret_cast<float4*>(p) + 1, make_float4(v[4], v[5], v[6], v[7]));
}
SB_DEVINL void st_stream_u4(void* p, uint4 v) { __stcs(reinterpret_cast<uint4*>(p), v); }
SB_DEVINL void st_stream_bf16(bf16* p, float v) {
  const unsigned short u = __bfloat16_as_ushort(__float2bfloat16_rn(v));
  asm volatile("st.global.cs.u16 [%0], %1;" ::"l"(p), "h"(u) : "memory");
}
SB_DEVINL uint4 pack8(const float (&v)[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
  return r;
}
SB_DEVINL void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7])
      : "r"(taddr)
      : "memory");
}

// =============================================================================================
// forward
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
  const int ring_bytes = p.ring * p.gc * Bp * 128;
  // the 128-row A read of the last ring slot overruns by (16 KB - stride) into this region
  const int wbytes = max(nchunks * WCHUNK, 16384 - Bp * 128);
  const GruSmem s = carve(smem_raw, ring_bytes, wbytes);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const uint32_t crank = cluster_rank(), csize = cluster_size();

  // ---- one-time setup: zero ring + weight region, stage the 48 weight rows, barriers, TMEM ----
  for (int k = tid; k < (ring_bytes + wbytes) / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(s.ring)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
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
  }
  if (tid == 0) {
    for (int i = 0; i < GRU_MAX_RING; ++i) {
      mbar_init(&s.full[i], 1);
      mbar_init(&s.empty[i], csize);
    }
    mbar_init(s.accfull, 1);
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(s.tmem_slot, 64);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();   // peers' barriers are initialised before anyone multicasts into them
  const uint32_t tmem_base = *s.tmem_slot;
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
      // this step's input projections do not depend on the recurrence: fetch them first
      float gi[3][GRU_UPT];
      if (active) {
        const float* g = p.gi + ((long long)t * Bp + row) * (p.ndir * 3 * H) + dir * 3 * H + ju;
#pragma unroll
        for (int gg = 0; gg < 3; ++gg) ld8(g + gg * H, gi[gg]);
      }
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
      float hn[GRU_UPT], rr[GRU_UPT], zz[GRU_UPT], nn[GRU_UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) {
          rr[jj] = fast_sigmoid(gi[0][jj] + acc[0][jj] + bias[0][jj]);
          zz[jj] = fast_sigmoid(gi[1][jj] + acc[1][jj] + bias[1][jj]);
          hn[jj] = acc[2][jj] + bias[2][jj];
          nn[jj] = fast_tanh(gi[2][jj] + rr[jj] * hn[jj]);
          hprev[jj] = (1.f - zz[jj]) * nn[jj] + zz[jj] * hprev[jj];
        }
        // critical path: only the bf16 h_t that the other CTAs gather next step
        *reinterpret_cast<uint4*>(p.xn + m * D + dir * H + ju) = pack8(hprev);
        if (tid == 0) GRU_STAMP(5);
        fence_proxy_async_global();   // generic writes -> other CTAs' TMA reads
        if (tid == 0) GRU_STAMP(6);
      }
      epi_barrier();
      if (tid == 0) {
        GRU_STAMP(7);
        grid_arrive(ctr);          // release: cumulative over the CTA's writes ordered by bar.sync
        GRU_STAMP(9);
      }
      // off the critical path: fp32 state, saved gates
      if (active) {
        st8(p.y + m * D + dir * H + ju, hprev);
        if (p.gates) {
          float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
          st8(go, rr);
          st8(go + H, zz);
          st8(go + 2 * H, nn);
          st8(go + 3 * H, hn);
        }
      }
      if (tid == 0) GRU_STAMP(10);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while peers may still signal its barriers
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 64);
  }
}

// =============================================================================================
// backward (reverse of the forward time order of each direction)
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
  const int ring_bytes = p.ring * p.gc * Bp * 128;
  const int wbytes = max(nchunks * WCHUNK, 16384 - Bp * 128);
  const GruSmem s = carve(smem_raw, ring_bytes, wbytes);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const uint32_t crank = cluster_rank(), csize = cluster_size();

  for (int k = tid; k < (ring_bytes + wbytes) / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(s.ring)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
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
  }
  if (tid == 0) {
    for (int i = 0; i < GRU_MAX_RING; ++i) {
      mbar_init(&s.full[i], 1);
      mbar_init(&s.empty[i], csize);
    }
    mbar_init(s.accfull, 1);
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(s.tmem_slot, 32);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();
  const uint32_t tmem_base = *s.tmem_slot;
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
    float db_r[GRU_UPT], db_z[GRU_UPT], db_n[GRU_UPT], db_hn[GRU_UPT];
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      dh_rec[jj] = 0.f; db_r[jj] = 0.f; db_z[jj] = 0.f; db_n[jj] = 0.f; db_hn[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      // forward order of dir 0 is t=0..T-1, so its backward order is T-1..0; dir 1 mirrored
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;       // time index of h_{prev} in forward order
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + row;
      // ---- saved activations of this step: independent of the recurrence, fetched first ----
      float rr[GRU_UPT], zz[GRU_UPT], nn[GRU_UPT], hn[GRU_UPT], dh[GRU_UPT], hp[GRU_UPT];
      if (active) {
        const float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
        ld8(go, rr);
        ld8(go + H, zz);
        ld8(go + 2 * H, nn);
        ld8(go + 3 * H, hn);
        ld8(p.dy + m * D + dir * H + ju, dh);
        if (has_prev) {
          ld8(p.y + ((long long)tp * Bp + row) * D + dir * H + ju, hp);
        } else {
#pragma unroll
          for (int jj = 0; jj < GRU_UPT; ++jj) hp[jj] = 0.f;
        }
      }
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
      float dr[GRU_UPT], dz[GRU_UPT], dn[GRU_UPT], dnr[GRU_UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) {
          const float g = dh[jj] + dh_rec[jj];
          dn[jj] = g * (1.f - zz[jj]) * (1.f - nn[jj] * nn[jj]);
          dz[jj] = g * (hp[jj] - nn[jj]) * zz[jj] * (1.f - zz[jj]);
          dr[jj] = dn[jj] * hn[jj] * rr[jj] * (1.f - rr[jj]);
          dnr[jj] = dn[jj] * rr[jj];
          dh_rec[jj] = g * zz[jj];      // direct path h_{t-1} -> h_t; the W_hh path is added next step
          db_r[jj] += dr[jj];
          db_z[jj] += dz[jj];
          db_n[jj] += dn[jj];
          db_hn[jj] += dnr[jj];
        }
        // critical path: the exchange rows [dr | dz | dn*r] every CTA gathers for the product
        if (step + 1 < T) {
          bf16* x = xb + (long long)row * K3 + ju;
          *reinterpret_cast<uint4*>(x) = pack8(dr);
          *reinterpret_cast<uint4*>(x + H) = pack8(dz);
          *reinterpret_cast<uint4*>(x + 2 * H) = pack8(dnr);
          if (tid == 0) GRU_STAMP(5);
          fence_proxy_async_global();
          if (tid == 0) GRU_STAMP(6);
        }
      }
      if (step + 1 < T) {
        epi_barrier();
        if (tid == 0) {
          GRU_STAMP(7);
          grid_arrive(ctr);
          GRU_STAMP(9);
        }
      }
      // ---- off the critical path: operands of the dX / dW GEMMs ----
      if (active) {
        bf16* o = p.dgi + m * (p.ndir * K3) + dir * K3 + ju;
        st_stream_u4(o, pack8(dr));
        st_stream_u4(o + H, pack8(dz));
        st_stream_u4(o + 2 * H, pack8(dn));
        st_stream_u4(p.dghn + m * D + dir * H + ju, pack8(dnr));
      }
      if (tid == 0) GRU_STAMP(10);
    }
    // ---- bias gradients: reduce the per-batch-row partial sums over the CTA ----
    epi_barrier();
    float* red = s.scratch;  // [64]: r(16) z(16) n(16) hn(16)
    if (tid < 64) red[tid] = 0.f;
    epi_barrier();
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      const float a = warp_sum(active ? db_r[jj] : 0.f);
      const float b = warp_sum(active ? db_z[jj] : 0.f);
      const float c = warp_sum(active ? db_n[jj] : 0.f);
      const float d = warp_sum(active ? db_hn[jj] : 0.f);
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

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 32);
  }
}

// =============================================================================================
// backward, K-split variant: the 4 CTAs of a cluster jointly own 64 hidden units.
//
// The plain backward kernel makes every CTA gather ALL of dgh_t (Bp x 3H bf16 = 384 KB at the
// north-star size) every step; with 96 KB of weights resident only 128 KB can be in flight, so
// the gather alone costs ~9 us of the 15.8 us step.  Here CTA r of a cluster contracts only the
// r-th QUARTER of the K = 3H dimension, for all 64 units of its cluster:
//     D_r[batch x 64] = dgh_t[:, quarter r] * W_hh[quarter r, 64 units]          (96 KB gathered)
// and the four partial products are reduce-scattered through distributed shared memory: each
// epilogue thread pushes the three 8-float slices that belong to peer CTAs with st.shared::cluster
// and arrives (release.cluster) on the peer's mbarrier; the owner adds the three slices it received
// to its own.  12 KB of DSMEM traffic replaces 288 KB of L2 reads per CTA per step.
// Requires cluster size 4, H % 256 == 0.
// =============================================================================================
static constexpr int KS = 4;

SB_DEVINL uint32_t mapa_shared(uint32_t local_addr, uint32_t peer) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(peer));
  return r;
}
SB_DEVINL void st_cluster_f4(uint32_t raddr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(raddr), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
SB_DEVINL void mbar_arrive_remote_release(uint32_t raddr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(raddr)
               : "memory");
}
SB_DEVINL void mbar_wait_acquire_cluster(uint64_t* bar, uint32_t parity) {
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
  constexpr int WCHUNK = 64 * 128;                    // 64 rows (units) x 64 bf16
  const int stride = Bp * 128;
  const int ring_bytes = nchunks * stride;            // the whole quarter is resident
  const int wbytes = nchunks * WCHUNK;
  // carve: ring | weights | recv | barriers
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* ring = base;
  uint8_t* wtile = ring + ring_bytes;
  float* recv = reinterpret_cast<float*>(wtile + wbytes);          // [KS][Bp][16] from peer src
  float* stage = recv + KS * Bp * 16;                              // [KS][Bp][16] for peer dst
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage + KS * Bp * 16);
  uint64_t* full = bars;          // [4] groups
  uint64_t* accfull = bars + 4;
  uint64_t* recvbar = bars + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const int gc = (nchunks % 4 == 0) ? 4 : ((nchunks % 3 == 0) ? 3 : ((nchunks % 2 == 0) ? 2 : 1));
  const int ngroups = nchunks / gc;                   // <= 4 for H <= 1024 ... checked on host

  for (int k = tid; k < (ring_bytes + wbytes + 2 * KS * Bp * 64) / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(base)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
    // resident operand: rows = the cluster's 64 units of W_hh^T, columns = this CTA's K quarter.
    // W_hh is read as stored ([3H][H]: the cluster's 64 units are 128 contiguous bytes of row k)
    // and transposed on the way into shared memory (once per launch)
    for (int k = tid; k < KQ * 8; k += GRU_THREADS) {
      const int kl = k >> 3, piece = k & 7;       // local k, 8-unit piece of the 64 units
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * K3 + (long long)crank * KQ + kl) * H + k0c + piece * 8);
      const unsigned short* e = reinterpret_cast<const unsigned short*>(&v);
      uint8_t* chunk = wtile + (kl >> 6) * WCHUNK + (kl & 7) * 2;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<unsigned short*>(
            chunk + sw128_offset((uint32_t)(piece * 8 + q), (uint32_t)((kl & 63) >> 3))) = e[q];
    }
  }
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&full[i], 1);
    mbar_init(accfull, 1);
    mbar_init(recvbar, 1);   // one local arrive.expect_tx per step; the peers' copies complete_tx
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(tmem_slot, 64);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();
  const uint32_t tmem_base = *tmem_slot;
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step) {
        grid_wait(ctr, (unsigned int)nC * (step + 1));   // dgh of this step is complete
        for (int g = 0; g < ngroups; ++g) {
          mbar_expect_tx(&full[g], (uint32_t)(stride * gc));
          for (int i = 0; i < gc; ++i) {
            const int c = g * gc + i;
            tma_load_2d(ring + c * stride, tm, &full[g], (int)crank * KQ + c * 64,
                        (step & 1) * Bp);
          }
        }
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(128, 64);
      for (int step = 0; step + 1 < T; ++step) {
        for (int g = 0; g < ngroups; ++g) {
          mbar_wait(&full[g], step & 1);
          tc_fence_after_sync();
          for (int i = 0; i < gc; ++i) {
            const int c = g * gc + i;
            const uint64_t da = umma_desc_sw128_kmajor(smem_u32(ring + c * stride));
            const uint64_t db = umma_desc_sw128_kmajor(smem_u32(wtile + c * WCHUNK));
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16_ss(tmem_base, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                           (c > 0 || kk > 0) ? 1u : 0u);
          }
        }
        umma_commit(accfull);
      }
    }
  } else {
    const int row = (warp & 3) * 32 + lane;
    const int uh = warp >> 2;
    const int ju = j0 + uh * GRU_UPT;
    const bool active = row < Bp;
    float dh_rec[GRU_UPT];
    float db_r[GRU_UPT], db_z[GRU_UPT], db_n[GRU_UPT], db_hn[GRU_UPT];
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      dh_rec[jj] = 0.f; db_r[jj] = 0.f; db_z[jj] = 0.f; db_n[jj] = 0.f; db_hn[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + row;
      float rr[GRU_UPT], zz[GRU_UPT], nn[GRU_UPT], hn[GRU_UPT], dh[GRU_UPT], hp[GRU_UPT];
      if (active) {
        const float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
        ld8(go, rr);
        ld8(go + H, zz);
        ld8(go + 2 * H, nn);
        ld8(go + 3 * H, hn);
        ld8(p.dy + m * D + dir * H + ju, dh);
        if (has_prev) {
          ld8(p.y + ((long long)tp * Bp + row) * D + dir * H + ju, hp);
        } else {
#pragma unroll
          for (int jj = 0; jj < GRU_UPT; ++jj) hp[jj] = 0.f;
        }
      }
      // ---- recurrent part of dL/dh_t: reduce-scatter of the four partial products ----
      if (step > 0) {
        mbar_wait(accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        float own[GRU_UPT];
        if (tid == 0) mbar_expect_tx(recvbar, (uint32_t)((KS - 1) * Bp * 16 * 4));
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
              float4* sp = reinterpret_cast<float4*>(stage + ((size_t)pr * Bp + row) * 16 +
                                                     uh * GRU_UPT);
              sp[0] = make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]),
                                  __uint_as_float(v[2]), __uint_as_float(v[3]));
              sp[1] = make_float4(__uint_as_float(v[4]), __uint_as_float(v[5]),
                                  __uint_as_float(v[6]), __uint_as_float(v[7]));
            }
            fence_proxy_async_smem();
            epi_barrier();
            if (tid == 0)
              bulk_s2peer(mapa_shared(smem_u32(recv + (size_t)crank * Bp * 16), pr),
                          stage + (size_t)pr * Bp * 16, (uint32_t)(Bp * 16 * 4),
                          mapa_shared(smem_u32(recvbar), pr));
          }
        }
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(recvbar, (step - 1) & 1);
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) dh_rec[jj] += own[jj];
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            if ((uint32_t)src == crank) continue;
            const float4* rp = reinterpret_cast<const float4*>(
                recv + ((size_t)src * Bp + row) * 16 + uh * GRU_UPT);
            const float4 a = rp[0], b = rp[1];
            dh_rec[0] += a.x; dh_rec[1] += a.y; dh_rec[2] += a.z; dh_rec[3] += a.w;
            dh_rec[4] += b.x; dh_rec[5] += b.y; dh_rec[6] += b.z; dh_rec[7] += b.w;
          }
        }
      }
      float dr[GRU_UPT], dz[GRU_UPT], dn[GRU_UPT], dnr[GRU_UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) {
          const float g = dh[jj] + dh_rec[jj];
          dn[jj] = g * (1.f - zz[jj]) * (1.f - nn[jj] * nn[jj]);
          dz[jj] = g * (hp[jj] - nn[jj]) * zz[jj] * (1.f - zz[jj]);
          dr[jj] = dn[jj] * hn[jj] * rr[jj] * (1.f - rr[jj]);
          dnr[jj] = dn[jj] * rr[jj];
          dh_rec[jj] = g * zz[jj];
          db_r[jj] += dr[jj];
          db_z[jj] += dz[jj];
          db_n[jj] += dn[jj];
          db_hn[jj] += dnr[jj];
        }
        if (step + 1 < T) {
          bf16* x = xb + (long long)row * K3 + ju;
          *reinterpret_cast<uint4*>(x) = pack8(dr);
          *reinterpret_cast<uint4*>(x + H) = pack8(dz);
          *reinterpret_cast<uint4*>(x + 2 * H) = pack8(dnr);
          if (tid == 0) GRU_STAMP(5);
          fence_proxy_async_global();
          if (tid == 0) GRU_STAMP(6);
        }
      }
      if (step + 1 < T) {
        epi_barrier();
        if (tid == 0) {
          GRU_STAMP(7);
          grid_arrive(ctr);
          GRU_STAMP(9);
        }
      }
      if (active) {
        bf16* o = p.dgi + m * (p.ndir * K3) + dir * K3 + ju;
        st_stream_u4(o, pack8(dr));
        st_stream_u4(o + H, pack8(dz));
        st_stream_u4(o + 2 * H, pack8(dn));
        st_stream_u4(p.dghn + m * D + dir * H + ju, pack8(dnr));
      }
      if (tid == 0) GRU_STAMP(10);
    }
#pragma unroll
    for (int jj = 0; jj < GRU_UPT; ++jj) {
      const float a = warp_sum(active ? db_r[jj] : 0.f);
      const float b = warp_sum(active ? db_z[jj] : 0.f);
      const float c = warp_sum(active ? db_n[jj] : 0.f);
      const float d = warp_sum(active ? db_hn[jj] : 0.f);
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

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 64);
  }
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
  const int ring_bytes = nchunks * stride;            // the whole quarter is resident
  const int wbytes = nchunks * WCHUNK;
  // carve: ring | weights | recv | barriers.  (The 128-row A read of the last chunk runs past the
  // ring into the weights: finite data, rows >= Bp are never used.)
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* ring = base;
  uint8_t* wtile = ring + ring_bytes;
  float* recv = reinterpret_cast<float*>(wtile + wbytes);          // [KS][Bp][48] from peer src
  float* stage = recv + KS * Bp * RW;                              // [KS][Bp][48] for peer dst
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage + KS * Bp * RW);
  uint64_t* full = bars;
  uint64_t* accfull = bars + 1;
  uint64_t* recvbar = bars + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  float* bias_s = reinterpret_cast<float*>(bars + 4);             // [48]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;

  for (int k = tid; k < (ring_bytes + wbytes + 2 * KS * Bp * RW * 4) / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(base)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
    // resident operand: rows = (gate, unit of the cluster), columns = this CTA's K quarter
    const int pieces_per_row = nchunks * 8;
    for (int k = tid; k < NCOL * pieces_per_row; k += GRU_THREADS) {
      const int r = k / pieces_per_row, pc = k % pieces_per_row;
      const int g = r / (KS * GRU_HC), u = r % (KS * GRU_HC);
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * 3 * H + (long long)g * H + k0c + u) * H + (long long)crank * KQ +
          pc * 8);
      *reinterpret_cast<uint4*>(wtile + (pc >> 3) * WCHUNK + sw128_offset(r, pc & 7)) = v;
    }
    if (tid < RW) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      bias_s[tid] = p.bhh[dir * 3 * H + g * H + j0 + jj];
    }
  }
  if (tid == 0) {
    mbar_init(full, 1);
    mbar_init(accfull, 1);
    mbar_init(recvbar, 1);   // one local arrive.expect_tx per step; the peers' copies complete_tx
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(tmem_slot, 256);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();
  const uint32_t tmem_base = *tmem_slot;
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
        mbar_expect_tx(full, (uint32_t)(stride * nchunks));
        for (int c = 0; c < nchunks; ++c)
          tma_load_2d(ring + c * stride, tm, full, (int)crank * KQ + c * 64, tp * Bp);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(128, NCOL);
      for (int step = 1; step < T; ++step) {
        mbar_wait(full, (step - 1) & 1);
        tc_fence_after_sync();
        for (int c = 0; c < nchunks; ++c) {
          const uint64_t da = umma_desc_sw128_kmajor(smem_u32(ring + c * stride));
          const uint64_t db = umma_desc_sw128_kmajor(smem_u32(wtile + c * WCHUNK));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16_ss(tmem_base, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                         (c > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(accfull);
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
      for (int jj = 0; jj < GRU_UPT; ++jj) bias[g][jj] = bias_s[g * GRU_HC + uh * GRU_UPT + jj];

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? step : (T - 1 - step);
      float gi[3][GRU_UPT];
      if (active) {
        const float* g = p.gi + ((long long)t * Bp + row) * (p.ndir * 3 * H) + dir * 3 * H + ju;
#pragma unroll
        for (int gg = 0; gg < 3; ++gg) ld8(g + gg * H, gi[gg]);
      }
      float acc[3][GRU_UPT];
#pragma unroll
      for (int gg = 0; gg < 3; ++gg)
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) acc[gg][jj] = 0.f;
      if (step > 0) {
        mbar_wait(accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        // ---- reduce-scatter of the four partial products.  The three slices that belong to
        // the peers go first, one at a time: TMEM -> registers -> local staging -> (named barrier)
        // -> ONE bulk copy into the peer's receive buffer, so the first copy is in flight while
        // the next slice is still being staged; the CTA's own slice is read last ----
        if (tid == 0) mbar_expect_tx(recvbar, (uint32_t)((KS - 1) * Bp * RW * 4));
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
              float* sp = stage + ((size_t)pr * Bp + row) * RW + uh * GRU_UPT;
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
              bulk_s2peer(mapa_shared(smem_u32(recv + (size_t)crank * Bp * RW), pr),
                          stage + (size_t)pr * Bp * RW, (uint32_t)(Bp * RW * 4),
                          mapa_shared(smem_u32(recvbar), pr));
          }
        }
        tc_fence_before_sync();
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            if ((uint32_t)src == crank) continue;
            const float* rp = recv + ((size_t)src * Bp + row) * RW + uh * GRU_UPT;
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
      float hn[GRU_UPT], rr[GRU_UPT], zz[GRU_UPT], nn[GRU_UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < GRU_UPT; ++jj) {
          rr[jj] = fast_sigmoid(gi[0][jj] + acc[0][jj] + bias[0][jj]);
          zz[jj] = fast_sigmoid(gi[1][jj] + acc[1][jj] + bias[1][jj]);
          hn[jj] = acc[2][jj] + bias[2][jj];
          nn[jj] = fast_tanh(gi[2][jj] + rr[jj] * hn[jj]);
          hprev[jj] = (1.f - zz[jj]) * nn[jj] + zz[jj] * hprev[jj];
        }
        // critical path: only the bf16 h_t that the other CTAs gather next step
        *reinterpret_cast<uint4*>(p.xn + m * D + dir * H + ju) = pack8(hprev);
        if (tid == 0) GRU_STAMP(5);
        fence_proxy_async_global();   // generic writes -> other CTAs' TMA reads
        if (tid == 0) GRU_STAMP(6);
      }
      epi_barrier();
      if (tid == 0) {
        GRU_STAMP(7);
        if (p.dbg && step == 20) p.dbg[1024 + blockIdx.x] = gtime();         // skew probe
        grid_arrive(ctr);
        GRU_STAMP(9);
      }
      if (active) {
        st8(p.y + m * D + dir * H + ju, hprev);
        if (p.gates) {
          float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
          st8(go, rr);
          st8(go + H, zz);
          st8(go + 2 * H, nn);
          st8(go + 3 * H, hn);
        }
      }
      if (tid == 0) GRU_STAMP(10);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 256);
  }
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
SB_DEVINL void ldu(const float* p, float (&v)[UPT]) {
  if constexpr (UPT == 2) {
    const float2 a = __ldcs(reinterpret_cast<const float2*>(p));
    v[0] = a.x; v[1] = a.y;
  } else {
    v[0] = __ldcs(p);
  }
}
template <int UPT>
SB_DEVINL void stu(float* p, const float (&v)[UPT]) {
  if constexpr (UPT == 2) __stcs(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
  else __stcs(p, v[0]);
}
template <int UPT>
SB_DEVINL void st_bf16u(bf16* p, const float (&v)[UPT]) {
  if constexpr (UPT == 2) {
    *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(v[0], v[1]);
  } else {
    *p = __float2bfloat16_rn(v[0]);
  }
}

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
  const int ring_bytes = nchunks * stride;            // the whole quarter is resident
  const int wbytes = nchunks * WCHUNK;
  // carve: ring | weights | recv | stage | barriers.  The N-side read of the last chunk may run
  // up to 8 rows past the ring into the weights, and the 128-row M-side read of tile 1 runs 64
  // rows past its 64 valid ones (into the next chunk / the receive buffer): both only feed
  // accumulator columns / lanes that are never read.
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* ring = base;
  uint8_t* wtile = ring + ring_bytes;
  float* recv = reinterpret_cast<float*>(wtile + wbytes);          // [KS src][48][P]
  float* stage = recv + KS * slice;                                // [KS-1 dst][48][P]
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage + (KS - 1) * slice);
  uint64_t* full = bars;
  uint64_t* accfull = bars + 1;
  uint64_t* recvbar = bars + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  float* bias_s = reinterpret_cast<float*>(bars + 4);             // [48]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;

  for (int k = tid; k < (ring_bytes + wbytes + (2 * KS - 1) * slice * 4) / 16; k += GRU_THREADS)
    reinterpret_cast<uint4*>(base)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
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
      *reinterpret_cast<uint4*>(wtile + (pc >> 3) * WCHUNK + sw128_offset(r, pc & 7)) = v;
    }
    if (tid < RW) {
      const int g = tid / GRU_HC, jj = tid % GRU_HC;
      bias_s[tid] = p.bhh[dir * 3 * H + g * H + j0 + jj];
    }
  }
  if (tid == 0) {
    mbar_init(full, 1);
    mbar_init(accfull, 1);
    mbar_init(recvbar, 1);   // one local arrive.expect_tx per step; the peers' copies complete_tx
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(tmem_slot, 128);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();
  const uint32_t tmem_base = *tmem_slot;
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
        mbar_expect_tx(full, (uint32_t)(stride * nchunks));
        for (int c = 0; c < nchunks; ++c)
          tma_load_2d(ring + c * stride, tm, full, (int)crank * KQ + c * 64, tp * Bp);
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(128, (uint32_t)NB);
      for (int step = 1; step < T; ++step) {
        mbar_wait(full, (step - 1) & 1);
        tc_fence_after_sync();
        for (int c = 0; c < nchunks; ++c) {
          const uint64_t da0 = umma_desc_sw128_kmajor(smem_u32(wtile + c * WCHUNK));
          const uint64_t da1 = umma_desc_sw128_kmajor(smem_u32(wtile + c * WCHUNK + 128 * 128));
          const uint64_t db = umma_desc_sw128_kmajor(smem_u32(ring + c * stride));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
            umma_bf16_ss(tmem_base, da0 + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc, acc);
            umma_bf16_ss(tmem_base + 64, da1 + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                         acc);
          }
        }
        umma_commit(accfull);
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
    float* dst0 = (q0 == 0 ? recv + crank * slice : stage + (q0 - 1) * slice) + lane * P;
    float* dst1 = (q1 == 0 ? recv + crank * slice : stage + (q1 - 1) * slice) +
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
      for (int jj = 0; jj < UPT; ++jj) bias[g][jj] = active ? bias_s[g * GRU_HC + u0 + jj] : 0.f;

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? step : (T - 1 - step);
      float gi[3][UPT];
      if (active) {
        const float* g = p.gi + ((long long)t * Bp + b) * (p.ndir * 3 * H) + dir * 3 * H + ju;
#pragma unroll
        for (int gg = 0; gg < 3; ++gg) ldu<UPT>(g + gg * H, gi[gg]);
      }
      float acc[3][UPT];
#pragma unroll
      for (int gg = 0; gg < 3; ++gg)
#pragma unroll
        for (int jj = 0; jj < UPT; ++jj) acc[gg][jj] = 0.f;
      if (step > 0) {
        mbar_wait(accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        if (tid == 0) mbar_expect_tx(recvbar, (uint32_t)((KS - 1) * slice * 4));
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
          bulk_s2peer(mapa_shared(smem_u32(recv + (size_t)crank * slice), pr),
                      stage + (size_t)(warp - 1) * slice, (uint32_t)(slice * 4),
                      mapa_shared(smem_u32(recvbar), pr));
        }
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            const float* rp = recv + (size_t)src * slice + u0 * P + b;
#pragma unroll
            for (int gg = 0; gg < 3; ++gg)
#pragma unroll
              for (int jj = 0; jj < UPT; ++jj) acc[gg][jj] += rp[(gg * GRU_HC + jj) * P];
          }
        }
      }
      const long long m = (long long)t * Bp + b;
      float hn[UPT], rr[UPT], zz[UPT], nn[UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < UPT; ++jj) {
          rr[jj] = fast_sigmoid(gi[0][jj] + acc[0][jj] + bias[0][jj]);
          zz[jj] = fast_sigmoid(gi[1][jj] + acc[1][jj] + bias[1][jj]);
          hn[jj] = acc[2][jj] + bias[2][jj];
          nn[jj] = fast_tanh(gi[2][jj] + rr[jj] * hn[jj]);
          hprev[jj] = (1.f - zz[jj]) * nn[jj] + zz[jj] * hprev[jj];
        }
        // critical path: only the bf16 h_t that the other CTAs gather next step
        st_bf16u<UPT>(p.xn + m * D + dir * H + ju, hprev);
        if (tid == 0) GRU_STAMP(5);
        fence_proxy_async_global();   // generic writes -> other CTAs' TMA reads
        if (tid == 0) GRU_STAMP(6);
      }
      epi_barrier();
      if (tid == 0) {
        GRU_STAMP(7);
        if (p.dbg && step == 20) p.dbg[1024 + blockIdx.x] = gtime();         // skew probe
        grid_arrive(ctr);
        GRU_STAMP(9);
      }
      if (active) {
        stu<UPT>(p.y + m * D + dir * H + ju, hprev);
        if (p.gates) {
          float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
          stu<UPT>(go, rr);
          stu<UPT>(go + H, zz);
          stu<UPT>(go + 2 * H, nn);
          stu<UPT>(go + 3 * H, hn);
        }
      }
      if (tid == 0) GRU_STAMP(10);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 128);
  }
}

// =============================================================================================
// backward, K split with the accumulator TRANSPOSED (see gru_fwd_kt_kernel):
//     D^T[64 units x Bp] = W_hh^T[64 units of the cluster, quarter r of 3H] * dgh[:, quarter r]^T
// The weight tile is the one of gru_bwd_ks_kernel (its 64 rows are already grouped by owner:
// rows 16q..16q+15 belong to CTA q of the cluster); an accumulator lane is a unit, so its row
// of Bp partial sums goes to exactly one peer, and the elementwise work runs on all 256
// epilogue threads (thread = batch row x UPT units).
// =============================================================================================
template <int UPT>
SB_DEVINL void st_stream_bf16u(bf16* p, const float (&v)[UPT]) {
  if constexpr (UPT == 2) {
    __stcs(reinterpret_cast<unsigned int*>(p), pack_bf16x2(v[0], v[1]));
  } else {
    st_stream_bf16(p, v[0]);
  }
}

template <int UPT>
__global__ void __launch_bounds__(GRU_THREADS, 1)
gru_bwd_kt_kernel(const __grid_constant__ CUtensorMap tm_d0,
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
  constexpr int WCHUNK = 64 * 128;                    // 64 rows (units) x 64 bf16
  const int P = Bp + 4;                               // pitch of a staged row (floats)
  const int slice = GRU_HC * P;                       // floats per (source, owner) slice
  const int NB = (Bp + 15) & ~15;
  const int stride = Bp * 128;
  const int ring_bytes = nchunks * stride;            // the whole quarter is resident
  const int wbytes = nchunks * WCHUNK;
  // carve: ring | weights | recv | stage | barriers.  The 128-row M-side read covers the next
  // weight chunk (last chunk: the receive buffer) with its lanes 64..127, which are never read.
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* ring = base;
  uint8_t* wtile = ring + ring_bytes;
  float* recv = reinterpret_cast<float*>(wtile + wbytes);          // [KS src][16][P]
  float* stage = recv + KS * slice;                                // [KS-1 dst][16][P]
  float* pad_end = stage + (KS - 1) * slice;
  // the last chunk's 128-row read needs 8 KB after the weights: recv + stage cover it only for
  // large batches, so reserve it explicitly
  const int tail_floats = max(0, 2048 - (2 * KS - 1) * slice);
  uint64_t* bars = reinterpret_cast<uint64_t*>(pad_end + tail_floats);
  uint64_t* full = bars;          // [4] groups
  uint64_t* accfull = bars + 4;
  uint64_t* recvbar = bars + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = p.ndir * H;
  const CUtensorMap* tm = dir == 0 ? &tm_d0 : &tm_d1;
  const int gc = (nchunks % 4 == 0) ? 4 : ((nchunks % 3 == 0) ? 3 : ((nchunks % 2 == 0) ? 2 : 1));
  const int ngroups = nchunks / gc;                   // <= 4 for H <= 1024 ... checked on host

  for (int k = tid; k < (ring_bytes + wbytes + ((2 * KS - 1) * slice + tail_floats) * 4) / 16;
       k += GRU_THREADS)
    reinterpret_cast<uint4*>(base)[k] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
    // resident operand: see gru_bwd_ks_kernel
    for (int k = tid; k < KQ * 8; k += GRU_THREADS) {
      const int kl = k >> 3, piece = k & 7;       // local k, 8-unit piece of the 64 units
      const uint4 v = *reinterpret_cast<const uint4*>(
          p.whh + ((long long)dir * K3 + (long long)crank * KQ + kl) * H + k0c + piece * 8);
      const unsigned short* e = reinterpret_cast<const unsigned short*>(&v);
      uint8_t* chunk = wtile + (kl >> 6) * WCHUNK + (kl & 7) * 2;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<unsigned short*>(
            chunk + sw128_offset((uint32_t)(piece * 8 + q), (uint32_t)((kl & 63) >> 3))) = e[q];
    }
  }
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&full[i], 1);
    mbar_init(accfull, 1);
    mbar_init(recvbar, 1);
    mbar_fence_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 8) tmem_alloc(tmem_slot, 64);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  cluster_sync_all();
  const uint32_t tmem_base = *tmem_slot;
  unsigned int* ctr = p.barrier + dir * 32;   // one L2 line per direction

  if (warp == 9) {
    if (lane == 0) {
      for (int step = 0; step + 1 < T; ++step) {
        grid_wait(ctr, (unsigned int)nC * (step + 1));   // dgh of this step is complete
        GRU_STAMP(0);
        for (int g = 0; g < ngroups; ++g) {
          mbar_expect_tx(&full[g], (uint32_t)(stride * gc));
          for (int i = 0; i < gc; ++i) {
            const int c = g * gc + i;
            tma_load_2d(ring + c * stride, tm, &full[g], (int)crank * KQ + c * 64,
                        (step & 1) * Bp);
          }
        }
        GRU_STAMP(1);
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(128, (uint32_t)NB);
      for (int step = 0; step + 1 < T; ++step) {
        for (int g = 0; g < ngroups; ++g) {
          mbar_wait(&full[g], step & 1);
          tc_fence_after_sync();
          for (int i = 0; i < gc; ++i) {
            const int c = g * gc + i;
            const uint64_t da = umma_desc_sw128_kmajor(smem_u32(wtile + c * WCHUNK));
            const uint64_t db = umma_desc_sw128_kmajor(smem_u32(ring + c * stride));
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16_ss(tmem_base, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc,
                           (c > 0 || kk > 0) ? 1u : 0u);
          }
        }
        umma_commit(accfull);
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
    float* dst0 = (q0 == 0 ? recv + crank * slice : stage + (q0 - 1) * slice) + (lane & 15) * P;
    // phase B: thread = (batch row b, UPT of the CTA's 16 units)
    const int b = tid % Bp, ug = tid / Bp;
    const bool active = ug * UPT < GRU_HC;
    const int u0 = ug * UPT;
    const int ju = j0 + u0;
    float dh_rec[UPT];
    float db_r[UPT], db_z[UPT], db_n[UPT], db_hn[UPT];
#pragma unroll
    for (int jj = 0; jj < UPT; ++jj) {
      dh_rec[jj] = 0.f; db_r[jj] = 0.f; db_z[jj] = 0.f; db_n[jj] = 0.f; db_hn[jj] = 0.f;
    }

    for (int step = 0; step < T; ++step) {
      const int t = dir == 0 ? (T - 1 - step) : step;
      const int tp = dir == 0 ? t - 1 : t + 1;
      const bool has_prev = dir == 0 ? (t > 0) : (t < T - 1);
      bf16* xb = p.xchg + ((long long)(dir * 2 + (step & 1)) * Bp) * K3;
      const long long m = (long long)t * Bp + b;
      float rr[UPT], zz[UPT], nn[UPT], hn[UPT], dh[UPT], hp[UPT];
      if (active) {
        const float* go = p.gates + ((m * p.ndir + dir) * 4) * H + ju;
        ldu<UPT>(go, rr);
        ldu<UPT>(go + H, zz);
        ldu<UPT>(go + 2 * H, nn);
        ldu<UPT>(go + 3 * H, hn);
        ldu<UPT>(p.dy + m * D + dir * H + ju, dh);
        if (has_prev) {
          ldu<UPT>(p.y + ((long long)tp * Bp + b) * D + dir * H + ju, hp);
        } else {
#pragma unroll
          for (int jj = 0; jj < UPT; ++jj) hp[jj] = 0.f;
        }
      }
      if (step > 0) {
        mbar_wait(accfull, (step - 1) & 1);
        if (tid == 0) GRU_STAMP(3);
        tc_fence_after_sync();
        if (tid == 0) mbar_expect_tx(recvbar, (uint32_t)((KS - 1) * slice * 4));
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
          bulk_s2peer(mapa_shared(smem_u32(recv + (size_t)crank * slice), pr),
                      stage + (size_t)(warp - 1) * slice, (uint32_t)(slice * 4),
                      mapa_shared(smem_u32(recvbar), pr));
        }
        if (tid == 0) GRU_STAMP(4);
        mbar_wait(recvbar, (step - 1) & 1);
        if (active) {
#pragma unroll
          for (int src = 0; src < KS; ++src) {
            const float* rp = recv + (size_t)src * slice + u0 * P + b;
#pragma unroll
            for (int jj = 0; jj < UPT; ++jj) dh_rec[jj] += rp[jj * P];
          }
        }
      }
      float dr[UPT], dz[UPT], dn[UPT], dnr[UPT];
      if (active) {
#pragma unroll
        for (int jj = 0; jj < UPT; ++jj) {
          const float g = dh[jj] + dh_rec[jj];
          dn[jj] = g * (1.f - zz[jj]) * (1.f - nn[jj] * nn[jj]);
          dz[jj] = g * (hp[jj] - nn[jj]) * zz[jj] * (1.f - zz[jj]);
          dr[jj] = dn[jj] * hn[jj] * rr[jj] * (1.f - rr[jj]);
          dnr[jj] = dn[jj] * rr[jj];
          dh_rec[jj] = g * zz[jj];
          db_r[jj] += dr[jj];
          db_z[jj] += dz[jj];
          db_n[jj] += dn[jj];
          db_hn[jj] += dnr[jj];
        }
        if (step + 1 < T) {
          bf16* x = xb + (long long)b * K3 + ju;
          st_bf16u<UPT>(x, dr);
          st_bf16u<UPT>(x + H, dz);
          st_bf16u<UPT>(x + 2 * H, dnr);
          if (tid == 0) GRU_STAMP(5);
          fence_proxy_async_global();
          if (tid == 0) GRU_STAMP(6);
        }
      }
      if (step + 1 < T) {
        epi_barrier();
        if (tid == 0) {
          GRU_STAMP(7);
          grid_arrive(ctr);
          GRU_STAMP(9);
        }
      }
      if (active) {
        bf16* o = p.dgi + m * (p.ndir * K3) + dir * K3 + ju;
        st_stream_bf16u<UPT>(o, dr);
        st_stream_bf16u<UPT>(o + H, dz);
        st_stream_bf16u<UPT>(o + 2 * H, dn);
        st_stream_bf16u<UPT>(p.dghn + m * D + dir * H + ju, dnr);
      }
      if (tid == 0) GRU_STAMP(10);
    }
    if (active) {
#pragma unroll
      for (int jj = 0; jj < UPT; ++jj) {
        const int bi = dir * K3 + ju + jj;
        atomicAdd(p.dbih + bi, db_r[jj]);
        atomicAdd(p.dbih + bi + H, db_z[jj]);
        atomicAdd(p.dbih + bi + 2 * H, db_n[jj]);
        atomicAdd(p.dbhh + bi, db_r[jj]);
        atomicAdd(p.dbhh + bi + H, db_z[jj]);
        atomicAdd(p.dbhh + bi + 2 * H, db_hn[jj]);
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 64);
  }
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, long long rows, long long cols,
                      long long ld, int box_rows);

// chunks are grouped gc per mbarrier pair (gc = largest of 4,3,2,1 dividing nchunks); ring = the
// largest divisor of ngroups (<= GRU_MAX_RING) whose slots fit next to the resident weights
static int gru_ring_slots(int wbytes, int Bp, int nchunks, int* gc_out, size_t* smem_bytes) {
  int gc = 1;
  for (int g = 4; g >= 1; --g)
    if (nchunks % g == 0) { gc = g; break; }
  const int ngroups = nchunks / gc;
  const int slot = gc * Bp * 128;
  const int fixed = wbytes + 1024 /*align*/ + (2 * GRU_MAX_RING + 2) * 8 + 256 /*scratch*/ + 64;
  int fit = (227 * 1024 - fixed) / slot;
  if (fit > GRU_MAX_RING) fit = GRU_MAX_RING;
  int ring = -1;
  for (int r = fit; r >= 1; --r)
    if (ngroups % r == 0) { ring = r; break; }
  if (ring < 1) {
    if (gc == 1) return -1;
    // fall back to single-chunk groups
    gc = 1;
    fit = (227 * 1024 - fixed) / (Bp * 128);
    if (fit > GRU_MAX_RING) fit = GRU_MAX_RING;
    for (int r = fit; r >= 1; --r)
      if (nchunks % r == 0) { ring = r; break; }
    if (ring < 1) return -1;
  }
  *gc_out = gc;
  *smem_bytes = (size_t)fixed + (size_t)ring * gc * Bp * 128;
  return ring;
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

extern "C" int sb_gru_fwd_workspace_size(int Bp, int H, int ndir, size_t* bytes) {
  if (!bytes || Bp <= 0 || H <= 0 || (ndir != 1 && ndir != 2)) return SB_ERR_INVALID;
  (void)Bp;
  *bytes = GRU_WS_COUNTERS;      // the forward kernels exchange h_t through xn itself
  return SB_OK;
}

extern "C" int sb_gru_fwd(const float* gi, const void* whh_bf16, const float* bhh, float* y,
                          void* xn_bf16, float* gates, void* workspace, size_t workspace_bytes,
                          int T, int Bp, int H, int ndir, void* stream_) {
  int rc = gru_check(T, Bp, H, ndir);
  if (rc != SB_OK) return rc;
  if (!gi || !whh_bf16 || !bhh || !y || !xn_bf16 || !workspace) return SB_ERR_INVALID;
  size_t need = 0;
  sb_gru_fwd_workspace_size(Bp, H, ndir, &need);
  if (workspace_bytes < need) return SB_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int nchunks = (H + 63) / 64;
  const int nC = H / GRU_HC;
  if (cudaMemsetAsync(workspace, 0, need, stream) != cudaSuccess) return SB_ERR_CUDA;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  unsigned int* barrier = reinterpret_cast<unsigned int*>(ws);
  int gc = 1;
  size_t smem = 0;
  const int ring =
      gru_ring_slots(std::max(nchunks * 48 * 128, 16384 - Bp * 128), Bp, nchunks, &gc, &smem);
  if (ring < 0) return SB_ERR_UNSUPPORTED;

  // ---- preferred: K-split over 4-CTA clusters (H % 256 == 0, batch rows <= 64) ----
  if (H % 256 == 0 && nC % KS == 0 && Bp <= 64) {
    const int nq = H / KS / 64;
    const size_t ks_smem = (size_t)nq * Bp * 128 + (size_t)nq * 192 * 128 +
                           (size_t)2 * KS * Bp * 48 * 4 + 1024 + 512;
    if (ks_smem <= 227 * 1024) {
      GruFwdParams q;
      q.gi = gi; q.whh = reinterpret_cast<const bf16*>(whh_bf16); q.bhh = bhh; q.y = y;
      q.xn = reinterpret_cast<bf16*>(xn_bf16); q.gates = gates;
      q.barrier = barrier; q.T = T; q.Bp = Bp; q.H = H; q.ndir = ndir;
      q.dbg = g_gru_dbg; q.ring = nq; q.gc = 1;
      CUtensorMap tq[2];
      for (int d = 0; d < 2; ++d) {
        const int dd = d < ndir ? d : 0;
        rc = make_tmap_bf16_2d(&tq[d], q.xn + (size_t)dd * H, (long long)T * Bp, H,
                               (long long)ndir * H, Bp);
        if (rc != SB_OK) return rc;
      }
      void* kargs[] = {(void*)&tq[0], (void*)&tq[1], (void*)&q};
      const size_t kt_smem = (size_t)nq * Bp * 128 + (size_t)nq * 192 * 128 +
                             (size_t)(2 * KS - 1) * 48 * (Bp + 4) * 4 + 1024 + 512;
      if (gru_use_kt(Bp, false) && kt_smem <= 227 * 1024) {
        const void* kt = Bp > 16 ? (const void*)gru_fwd_kt_kernel<2>
                                 : (const void*)gru_fwd_kt_kernel<1>;
        rc = gru_launch(kt, ndir * nC, nC, KS, KS, kt_smem, kargs, stream);
        if (rc == SB_OK) return SB_OK;
      }
      rc = gru_launch((const void*)gru_fwd_ks_kernel, ndir * nC, nC, KS, KS, ks_smem, kargs, stream);
      if (rc == SB_OK) return SB_OK;
    }
  }

  // ---- every other shape: each CTA gathers all of h_{t-1} (tensor-map TMA, cluster multicast) ----
  GruFwdParams p;
  p.gi = gi; p.whh = reinterpret_cast<const bf16*>(whh_bf16); p.bhh = bhh; p.y = y;
  p.xn = reinterpret_cast<bf16*>(xn_bf16);
  p.gates = gates; p.barrier = barrier; p.T = T; p.Bp = Bp; p.H = H; p.ndir = ndir;
  p.dbg = g_gru_dbg;
  p.ring = ring; p.gc = gc;
  CUtensorMap tm[2];
  for (int d = 0; d < 2; ++d) {
    const int dd = d < ndir ? d : 0;
    rc = make_tmap_bf16_2d(&tm[d], p.xn + (size_t)dd * H, (long long)T * Bp, H,
                           (long long)ndir * H, Bp);
    if (rc != SB_OK) return rc;
  }
  void* args[] = {(void*)&tm[0], (void*)&tm[1], (void*)&p};
  return gru_launch((const void*)gru_fwd_kernel, ndir * nC, nC, 4, 1, smem, args, stream);
}

extern "C" int sb_gru_bwd_workspace_size(int Bp, int H, int ndir, size_t* bytes) {
  if (!bytes || Bp <= 0 || H <= 0 || (ndir != 1 && ndir != 2)) return SB_ERR_INVALID;
  // counters + the double-buffered exchange of dgh_t (Bp x 3H bf16 per direction and parity; the
  // tile-major form of the K-split kernel rounds 3H up to whole 64-column chunks)
  const size_t k3p = (size_t)((3 * H + 63) / 64) * 64;
  *bytes = GRU_WS_COUNTERS + (size_t)ndir * 2 * Bp * k3p * sizeof(bf16) + 1024;
  return SB_OK;
}

extern "C" int sb_gru_bwd(const float* dy, const float* y, const float* gates,
                          const void* whh_bf16, void* dgi_bf16, void* dghn_bf16, float* dbih,
                          float* dbhh, void* workspace, size_t workspace_bytes, int T, int Bp,
                          int H, int ndir, void* stream_) {
  int rc = gru_check(T, Bp, H, ndir);
  if (rc != SB_OK) return rc;
  if (!dy || !y || !gates || !whh_bf16 || !dgi_bf16 || !dghn_bf16 || !dbih || !dbhh ||
      !workspace)
    return SB_ERR_INVALID;
  size_t need = 0;
  sb_gru_bwd_workspace_size(Bp, H, ndir, &need);
  if (workspace_bytes < need) return SB_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  GruBwdParams p;
  p.dy = dy; p.y = y; p.gates = gates; p.whh = reinterpret_cast<const bf16*>(whh_bf16);
  p.dgi = reinterpret_cast<bf16*>(dgi_bf16);
  p.dghn = reinterpret_cast<bf16*>(dghn_bf16);
  p.barrier = reinterpret_cast<unsigned int*>(ws);
  p.xchg = reinterpret_cast<bf16*>(ws + GRU_WS_COUNTERS);
  p.dbih = dbih; p.dbhh = dbhh; p.T = T; p.Bp = Bp; p.H = H; p.ndir = ndir;
  p.dbg = g_gru_dbg;
  const int K3 = 3 * H;
  const int nchunks = (K3 + 63) / 64;
  size_t smem = 0;
  const int nC_ = H / GRU_HC;
  // counters and barrier words start at zero; the exchange tiles too (columns past 3H of a
  // partial chunk are never written and must read as zero)
  if (cudaMemsetAsync(workspace, 0, need, stream) != cudaSuccess) return SB_ERR_CUDA;
  // ---- preferred: K-split over 4-CTA clusters ----
  if (H % 256 == 0 && nC_ % KS == 0 && (K3 / KS / 64) <= 16) {
    const int nq = K3 / KS / 64;
    const size_t ks_smem = (size_t)nq * Bp * 128 + (size_t)nq * 64 * 128 +
                           (size_t)2 * KS * Bp * 64 + 1024 + 256;
    if (ks_smem <= 227 * 1024) {
      CUtensorMap tq[2];
      for (int d = 0; d < 2; ++d) {
        const int dd = d < ndir ? d : 0;
        rc = make_tmap_bf16_2d(&tq[d], p.xchg + (size_t)dd * 2 * Bp * K3, 2LL * Bp, K3, K3, Bp);
        if (rc != SB_OK) return rc;
      }
      p.ring = nq; p.gc = 1;
      void* kargs[] = {(void*)&tq[0], (void*)&tq[1], (void*)&p};
      const size_t ex = (size_t)(2 * KS - 1) * GRU_HC * (Bp + 4) * 4;
      const size_t kt_smem = (size_t)nq * Bp * 128 + (size_t)nq * 64 * 128 +
                             std::max(ex, (size_t)8192) + 1024 + 256;
      if (gru_use_kt(Bp, true) && kt_smem <= 227 * 1024) {
        rc = gru_launch((const void*)gru_bwd_kt_kernel<1>, ndir * nC_, nC_, KS, KS, kt_smem, kargs,
                        stream);
        if (rc == SB_OK) return SB_OK;
      }
      rc = gru_launch((const void*)gru_bwd_ks_kernel, ndir * nC_, nC_, KS, KS, ks_smem, kargs,
                      stream);
      if (rc == SB_OK) return SB_OK;
    }
  }
  p.ring = gru_ring_slots(std::max(nchunks * 16 * 128, 16384 - Bp * 128), Bp, nchunks, &p.gc, &smem);
  if (p.ring < 0) return SB_ERR_UNSUPPORTED;
  // per direction: the two parity buffers stacked as [2*Bp rows][3H cols]
  CUtensorMap tm[2];
  for (int d = 0; d < 2; ++d) {
    const int dd = d < ndir ? d : 0;
    rc = make_tmap_bf16_2d(&tm[d], p.xchg + (size_t)dd * 2 * Bp * K3, 2LL * Bp, K3, K3, Bp);
    if (rc != SB_OK) return rc;
  }
  void* args[] = {(void*)&tm[0], (void*)&tm[1], (void*)&p};
  return gru_launch((const void*)gru_bwd_kernel, ndir * nC_, nC_, 4, 1, smem, args, stream);
}
