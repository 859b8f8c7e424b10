// Conv2d(+ReLU) front-end of the encoder as im2col + tensor-core GEMM.
//
// Replaces the cuDNN convolutions behind nn.Conv2d in Model.__init__/encode
// (speech/models/model.py:19-29,60-71): valid (padding 0) 2-D convolution over (time, freq) with
// kernel (kh, kw) and stride s in both dims, followed by ReLU; the stack's output is flattened
// channel-major to (B, T', C*F') (model.py:66-71).
//
// Layouts (all row-major):
//   activations between layers: "pixel-major channels-last"  P[(b*To + t)*Fo + f][c]  f32 =
//       exactly the C matrix of the GEMM; ReLU is applied by whoever READS it (so the
//       pre-activation sign is available to the backward mask);
//   im2col matrix A[m][(i*kw + j)*Ci + ci] bf16 (K padded to a multiple of 8 with zeros); the
//       weights are permuted to the same K order on the host side (40 K elements);
//   conv = sb_gemm_bf16_tn(A, Wp) + bias  on tcgen05.
// Backward: dC (pre-activation grad, bf16) -> dW^T = A^T dC (GEMM, both operands MN-major, split-K),
//   dA = dC Wp (GEMM), col2im as a GATHER (each input pixel sums its <= ceil(kh/s)*ceil(kw/s)
//   taps; no atomics) fused with the ReLU mask of the layer below.
// All kernels here are HBM-bound elementwise/gather kernels (algorithmic bytes = one read of the
// source + one write of the destination); the FLOPs run in gemm.cu.
#include "common.cuh"

#include "../../include/speech_b200.h"

namespace sb {

typedef __nv_bfloat16 bf16;

// ---- im2col ------------------------------------------------------------------------------------
// src: P[(b*Ti + ti)*Fi + fi][Ci] f32 (relu on read if `relu`), dst: A[M][Kp] bf16.
// One thread produces 8 consecutive K entries (one 16-byte store).  For Ci % 8 == 0 these are 8
// channels of one tap (two float4 loads); otherwise the scalar path is used per element.
__global__ void __launch_bounds__(256)
im2col_kernel(const float* __restrict__ src, const unsigned char* __restrict__ mask,
              float mscale, bf16* __restrict__ dst, int B, int Ti, int Fi, int Ci,
              int kh, int kw, int s, int To, int Fo, int Kp, int relu) {
  const int K = kh * kw * Ci;
  const int kvec = Kp >> 3;                       // 8-wide groups per row
  const long long M = (long long)B * To * Fo;
  const long long total = M * kvec;
  const bool vec = (Ci & 7) == 0;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    const long long m = idx / kvec;
    const int k0 = (int)(idx - m * kvec) << 3;
    const int f = (int)(m % Fo);
    const int bt = (int)(m / Fo);
    const int t = bt % To;
    const int b = bt / To;
    float v[8];
    if (vec && k0 < K) {
      const int ci = k0 % Ci;
      const int ij = k0 / Ci;
      const int j = ij % kw, i = ij / kw;
      const long long off = (((long long)b * Ti + (s * t + i)) * Fi + (s * f + j)) * Ci + ci;
      const float4* p = reinterpret_cast<const float4*>(src + off);
      const float4 a = __ldg(p), c = __ldg(p + 1);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
      if (relu) {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = fmaxf(v[e], 0.f);
      }
      if (mask) {   // dropout of the layer below: keep-byte per element, same layout as src
        const uint2 mk = __ldg(reinterpret_cast<const uint2*>(mask + off));
        const unsigned char* mb = reinterpret_cast<const unsigned char*>(&mk);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = mb[e] ? v[e] * mscale : 0.f;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = k0 + e;
        v[e] = 0.f;
        if (k < K) {
          const int ci = k % Ci;
          const int ij = k / Ci;
          const int j = ij % kw, i = ij / kw;
          const long long off = (((long long)b * Ti + (s * t + i)) * Fi + (s * f + j)) * Ci + ci;
          v[e] = __ldg(src + off);
          if (relu) v[e] = fmaxf(v[e], 0.f);
          if (mask) v[e] = mask[off] ? v[e] * mscale : 0.f;
        }
      }
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(dst + m * Kp + k0) = o;
  }
}

// ---- final relayout: C[(b*To+t)*Fo+f][c] -> out[b][t][c*Fo + f] with ReLU ------------------------
__global__ void __launch_bounds__(256)
relu_to_bct_kernel(const float* __restrict__ C, const unsigned char* __restrict__ mask,
                   float mscale, float* __restrict__ out, int B, int To, int Fo, int Co) {
  const long long total = (long long)B * To * Fo * Co;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    // idx enumerates the OUTPUT (f fastest) so that writes are coalesced
    const int f = (int)(idx % Fo);
    long long r = idx / Fo;
    const int c = (int)(r % Co);
    r /= Co;                       // r = b*To + t
    const long long src = (r * Fo + f) * Co + c;
    float v = fmaxf(__ldg(C + src), 0.f);
    if (mask) v = mask[src] ? v * mscale : 0.f;
    out[idx] = v;
  }
}

// ---- top of backward: dY[b][t][c*Fo+f] * (C > 0) -> dC[(b*To+t)*Fo+f][c] bf16, db[c] += ----------
__global__ void __launch_bounds__(256)
dconv_top_kernel(const float* __restrict__ dY, const float* __restrict__ C,
                 const unsigned char* __restrict__ mask, float mscale, bf16* __restrict__ dC,
                 float* __restrict__ db, int B, int To, int Fo, int Co) {
  extern __shared__ float dbs[];
  for (int c = threadIdx.x; c < Co; c += 256) dbs[c] = 0.f;
  __syncthreads();
  const long long total = (long long)B * To * Fo * Co;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    const int c = (int)(idx % Co);     // idx enumerates dC (c fastest)
    const long long m = idx / Co;
    const int f = (int)(m % Fo);
    const long long r = m / Fo;
    float g = __ldg(dY + (r * Co + c) * Fo + f);
    if (__ldg(C + idx) <= 0.f) g = 0.f;
    else if (mask) g = mask[idx] ? g * mscale : 0.f;
    dC[idx] = __float2bfloat16_rn(g);
    if (g != 0.f) atomicAdd(&dbs[c], g);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Co; c += 256)
    if (dbs[c] != 0.f) atomicAdd(db + c, dbs[c]);
}

// ---- col2im as a gather, fused with the ReLU mask of the layer below -----------------------------
// dA[m][(i*kw+j)*Ci + ci] f32 (ld = ldA) -> dCprev[(b*Ti+ti)*Fi+fi][ci] bf16 (masked by Pprev > 0)
// Each input pixel receives at most ceil(kh/s)*ceil(kw/s) taps.  All tap loads of a thread are
// issued before any is consumed (a loop with data-dependent `continue`s left ONE load in flight
// per thread and ran at 0.9 TB/s).
template <int MAXI, int MAXJ>
__global__ void __launch_bounds__(256)
col2im_relu_kernel(const float* __restrict__ dA, long long ldA, const float* __restrict__ Pprev,
                   const unsigned char* __restrict__ maskprev, float mscale,
                   bf16* __restrict__ dCprev, float* __restrict__ db, int B, int Ti, int Fi,
                   int Ci, int kh, int kw, int s, int To, int Fo) {
  extern __shared__ float dbs[];
  for (int c = threadIdx.x; c < Ci; c += 256) dbs[c] = 0.f;
  __syncthreads();
  const long long total = (long long)B * Ti * Fi * Ci;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    const int ci = (int)(idx % Ci);
    const int px = (int)(idx / Ci);
    const int fi = px % Fi;
    const int bt = px / Fi;
    const int ti = bt % Ti;
    const int b = bt / Ti;
    const float mask = __ldg(Pprev + idx);
    float v[MAXI * MAXJ];
#pragma unroll
    for (int a = 0; a < MAXI; ++a) {
      const int i = ti % s + a * s;
      const int t = (ti - i) / s;
      const bool okt = (i < kh) && (ti - i >= 0) && (t < To);
#pragma unroll
      for (int c = 0; c < MAXJ; ++c) {
        const int j = fi % s + c * s;
        const int f = (fi - j) / s;
        const bool ok = okt && (j < kw) && (fi - j >= 0) && (f < Fo);
        v[a * MAXJ + c] = 0.f;
        if (ok)
          v[a * MAXJ + c] =
              __ldcs(dA + (((long long)b * To + t) * Fo + f) * ldA + (i * kw + j) * Ci + ci);
      }
    }
    float g = 0.f;
#pragma unroll
    for (int e = 0; e < MAXI * MAXJ; ++e) g += v[e];
    if (mask <= 0.f) g = 0.f;
    else if (maskprev) g = maskprev[idx] ? g * mscale : 0.f;
    dCprev[idx] = __float2bfloat16_rn(g);
    if (g != 0.f) atomicAdd(&dbs[ci], g);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Ci; c += 256)
    if (dbs[c] != 0.f) atomicAdd(db + c, dbs[c]);
}

// Same gather with FOUR channels per thread (Ci % 4 == 0): 16-byte tap loads, a quarter of the
// index arithmetic per element (the scalar kernel was instruction-bound: 0.70 ms at 1.9 TB/s).
template <int MAXI, int MAXJ>
__global__ void __launch_bounds__(256)
col2im_relu_v4_kernel(const float* __restrict__ dA, long long ldA, const float* __restrict__ Pprev,
                      const unsigned char* __restrict__ maskprev, float mscale,
                      bf16* __restrict__ dCprev, float* __restrict__ db, int B, int Ti, int Fi,
                      int Ci, int kh, int kw, int s, int To, int Fo) {
  extern __shared__ float dbs[];
  for (int c = threadIdx.x; c < Ci; c += 256) dbs[c] = 0.f;
  __syncthreads();
  const int C4 = Ci >> 2;
  const long long total = (long long)B * Ti * Fi * C4;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    const int c4 = (int)(idx % C4);
    const int px = (int)(idx / C4);
    const int fi = px % Fi;
    const int bt = px / Fi;
    const int ti = bt % Ti;
    const int b = bt / Ti;
    const float4 mask = __ldg(reinterpret_cast<const float4*>(Pprev) + idx);
    float4 v[MAXI * MAXJ];
#pragma unroll
    for (int a = 0; a < MAXI; ++a) {
      const int i = ti % s + a * s;
      const int t = (ti - i) / s;
      const bool okt = (i < kh) && (ti - i >= 0) && (t < To);
#pragma unroll
      for (int c = 0; c < MAXJ; ++c) {
        const int j = fi % s + c * s;
        const int f = (fi - j) / s;
        const bool ok = okt && (j < kw) && (fi - j >= 0) && (f < Fo);
        v[a * MAXJ + c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok)
          v[a * MAXJ + c] = __ldcs(reinterpret_cast<const float4*>(
              dA + (((long long)b * To + t) * Fo + f) * ldA + (i * kw + j) * Ci + c4 * 4));
      }
    }
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int e = 0; e < MAXI * MAXJ; ++e) { g.x += v[e].x; g.y += v[e].y; g.z += v[e].z; g.w += v[e].w; }
    if (mask.x <= 0.f) g.x = 0.f;
    if (mask.y <= 0.f) g.y = 0.f;
    if (mask.z <= 0.f) g.z = 0.f;
    if (mask.w <= 0.f) g.w = 0.f;
    if (maskprev) {
      const uchar4 mk = reinterpret_cast<const uchar4*>(maskprev)[idx];
      g.x = mk.x ? g.x * mscale : 0.f; g.y = mk.y ? g.y * mscale : 0.f;
      g.z = mk.z ? g.z * mscale : 0.f; g.w = mk.w ? g.w * mscale : 0.f;
    }
    reinterpret_cast<uint2*>(dCprev)[idx] = make_uint2(pack_bf16x2(g.x, g.y), pack_bf16x2(g.z, g.w));
    if (g.x != 0.f) atomicAdd(&dbs[c4 * 4], g.x);
    if (g.y != 0.f) atomicAdd(&dbs[c4 * 4 + 1], g.y);
    if (g.z != 0.f) atomicAdd(&dbs[c4 * 4 + 2], g.z);
    if (g.w != 0.f) atomicAdd(&dbs[c4 * 4 + 3], g.w);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Ci; c += 256)
    if (dbs[c] != 0.f) atomicAdd(db + c, dbs[c]);
}

// Any tap count (runtime loops): the TIMIT recipes' second layer [*, 5, 32, 1] has 5 x 32 taps per
// input pixel, far beyond the unrolled instantiations above.  The inner loop over j is unrolled by
// 4 with the loads issued before their use, so 4 loads are in flight per thread.
__global__ void __launch_bounds__(256)
col2im_relu_generic_kernel(const float* __restrict__ dA, long long ldA,
                           const float* __restrict__ Pprev,
                           const unsigned char* __restrict__ maskprev, float mscale,
                           bf16* __restrict__ dCprev, float* __restrict__ db, int B, int Ti, int Fi,
                           int Ci, int kh, int kw, int s, int To, int Fo) {
  extern __shared__ float dbs[];
  for (int c = threadIdx.x; c < Ci; c += 256) dbs[c] = 0.f;
  __syncthreads();
  const long long total = (long long)B * Ti * Fi * Ci;
  for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * 256) {
    const int ci = (int)(idx % Ci);
    const int px = (int)(idx / Ci);
    const int fi = px % Fi;
    const int bt = px / Fi;
    const int ti = bt % Ti;
    const int b = bt / Ti;
    const float mask = __ldg(Pprev + idx);
    float g = 0.f;
    if (mask > 0.f) {
      for (int i = ti % s; i < kh && i <= ti; i += s) {
        const int t = (ti - i) / s;
        if (t >= To) continue;
        const float* rowp = dA + ((long long)b * To + t) * Fo * ldA + (long long)i * kw * Ci + ci;
        int j = fi % s;
        for (; j + 3 * s < kw && j + 3 * s <= fi; j += 4 * s) {
          float v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int f = (fi - j - u * s) / s;
            v[u] = f < Fo ? __ldcs(rowp + (long long)f * ldA + (j + u * s) * Ci) : 0.f;
          }
          g += (v[0] + v[1]) + (v[2] + v[3]);
        }
        for (; j < kw && j <= fi; j += s) {
          const int f = (fi - j) / s;
          if (f < Fo) g += __ldcs(rowp + (long long)f * ldA + j * Ci);
        }
      }
      if (maskprev) g = maskprev[idx] ? g * mscale : 0.f;
    }
    dCprev[idx] = __float2bfloat16_rn(g);
    if (g != 0.f) atomicAdd(&dbs[ci], g);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Ci; c += 256)
    if (dbs[c] != 0.f) atomicAdd(db + c, dbs[c]);
}

static int grid_for(long long total) {
  long long g = (total + 255) / 256;
  const long long cap = (long long)device_sm_count() * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace sb

using namespace sb;

extern "C" int sb_conv_im2col(const float* src, const void* mask_u8, float mscale,
                              void* dst_bf16, int B,
                              int Ti, int Fi, int Ci, int kh, int kw, int stride, int Kp,
                              int relu, void* stream_) {
  if (!src || !dst_bf16 || B <= 0 || Ci <= 0 || kh <= 0 || kw <= 0 || stride <= 0)
    return SB_ERR_INVALID;
  const int To = (Ti - kh) / stride + 1, Fo = (Fi - kw) / stride + 1;
  if (To <= 0 || Fo <= 0 || Kp < kh * kw * Ci) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const long long total = (long long)B * To * Fo * (Kp / 8);
  im2col_kernel<<<grid_for(total), 256, 0, stream>>>(
      src, reinterpret_cast<const unsigned char*>(mask_u8), mscale,
      reinterpret_cast<bf16*>(dst_bf16), B, Ti, Fi,
      Ci, kh, kw, stride, To, Fo, Kp, relu);
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}

extern "C" int sb_conv_relu_to_bct(const float* C, const void* mask_u8, float mscale,
                                   float* out, int B,
                                   int To, int Fo, int Co, void* stream_) {
  if (!C || !out || B <= 0 || To <= 0 || Fo <= 0 || Co <= 0) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  relu_to_bct_kernel<<<grid_for((long long)B * To * Fo * Co), 256, 0, stream>>>(
      C, reinterpret_cast<const unsigned char*>(mask_u8), mscale, out, B, To, Fo, Co);
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}

extern "C" int sb_conv_dtop(const float* dY, const float* C, const void* mask_u8, float mscale,
                            void* dC_bf16,
                            float* db, int B, int To, int Fo, int Co, void* stream_) {
  if (!dY || !C || !dC_bf16 || !db || B <= 0 || To <= 0 || Fo <= 0 || Co <= 0)
    return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  dconv_top_kernel<<<grid_for((long long)B * To * Fo * Co), 256, Co * sizeof(float), stream>>>(
      dY, C, reinterpret_cast<const unsigned char*>(mask_u8), mscale,
      reinterpret_cast<bf16*>(dC_bf16), db, B, To, Fo, Co);
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}

extern "C" int sb_conv_col2im_relu(const float* dA, long long ldA, const float* Pprev,
                                   const void* maskprev_u8, float mscale, void* dCprev_bf16,
                                   float* db, int B,
                                   int Ti, int Fi, int Ci, int kh, int kw, int stride,
                                   void* stream_) {
  if (!dA || !Pprev || !dCprev_bf16 || !db || B <= 0) return SB_ERR_INVALID;
  const int To = (Ti - kh) / stride + 1, Fo = (Fi - kw) / stride + 1;
  if (To <= 0 || Fo <= 0) return SB_ERR_INVALID;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int ni = (kh + stride - 1) / stride, nj = (kw + stride - 1) / stride;
  const int g = grid_for((long long)B * Ti * Fi * Ci);
  bf16* out = reinterpret_cast<bf16*>(dCprev_bf16);
  const size_t sm = Ci * sizeof(float);
  if ((long long)B * Ti * Fi >= (1LL << 31)) return SB_ERR_UNSUPPORTED;
#define SB_C2I(I, J)                                                                              \
  col2im_relu_kernel<I, J><<<g, 256, sm, stream>>>(                                                \
      dA, ldA, Pprev, reinterpret_cast<const unsigned char*>(maskprev_u8), mscale, out, db, B, Ti,  \
      Fi, Ci, kh, kw,                                                                                 \
      stride, To, Fo)
  // four channels per thread when the layout allows 16-byte tap loads
  const bool v4 = (Ci % 4 == 0) && (ldA % 4 == 0) && ((reinterpret_cast<uintptr_t>(dA) & 15) == 0) &&
                  ((reinterpret_cast<uintptr_t>(Pprev) & 15) == 0) &&
                  ((reinterpret_cast<uintptr_t>(dCprev_bf16) & 7) == 0) &&
                  (!maskprev_u8 || (reinterpret_cast<uintptr_t>(maskprev_u8) & 3) == 0);
  const int g4 = grid_for((long long)B * Ti * Fi * (Ci / 4));
#define SB_C2I4(I, J)                                                                             \
  col2im_relu_v4_kernel<I, J><<<g4, 256, sm, stream>>>(                                            \
      dA, ldA, Pprev, reinterpret_cast<const unsigned char*>(maskprev_u8), mscale, out, db, B, Ti,  \
      Fi, Ci, kh, kw, stride, To, Fo)
  if (v4 && ni <= 2 && nj <= 2) SB_C2I4(2, 2);
  else if (v4 && ni <= 3 && nj <= 4) SB_C2I4(3, 4);
  else if (ni <= 2 && nj <= 2) SB_C2I(2, 2);
  else if (ni <= 3 && nj <= 4) SB_C2I(3, 4);
  else if (ni <= 5 && nj <= 8) SB_C2I(5, 8);
  else
    col2im_relu_generic_kernel<<<g, 256, sm, stream>>>(
        dA, ldA, Pprev, reinterpret_cast<const unsigned char*>(maskprev_u8), mscale, out, db, B, Ti,
        Fi, Ci, kh, kw, stride, To, Fo);
#undef SB_C2I
#undef SB_C2I4
  return cudaGetLastError() == cudaSuccess ? SB_OK : SB_ERR_CUDA;
}
