// LayerNorm forward / backward (fp32 statistics, HBM-bound; vectorised, coalesced).
// Replaces nn.LayerNorm at helpers.py:17 (FeedForward), :32-33/:47-48 (PerceiverAttention norm_media /
// norm_latents), :105/:132 (PerceiverResampler.norm), :151/:184 (MaskedCrossAttention.norm) and the
// ViT ln_pre / ln_1 / ln_2 (open_clip, third party).  The forward writes the normalised rows as bf16 so
// they are the TMA-ready A operand of the following GEMM (the reference's autocast casts the fp32 LN
// output to bf16 inside nn.Linear -- same rounding point), and can write them at an offset/stride so the
// two LayerNorms of PerceiverAttention fill cat((x, latents), -2) (helpers.py:53) without a copy kernel.
// RMS = true is the RMSNorm variant (HF LlamaRMSNorm: no centring, no beta, y = gamma * (x * rstd)).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ofk_internal.h"
#include "ofk_ptx.cuh"

namespace ofk {

__device__ __forceinline__ long long map_row(int r, int rpg, int gstride, int goff) {
  if (rpg <= 0) return r;
  return (long long)(r / rpg) * gstride + goff + (r % rpg);
}

// One warp per row; each lane keeps NV float4 (columns (i*32 + lane)*4) in registers.
template <int NV, bool RMS = false>
__global__ void __launch_bounds__(128) ln_fwd_kernel(const float* __restrict__ x, long long ldx,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     float eps, int rows, int D, void* __restrict__ y, int y_is_f32,
                                                     long long ldy, int rpg, int gstride, int goff,
                                                     float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + (long long)row * ldx;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < D) {
      v[i] = *reinterpret_cast<const float4*>(xr + c);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    } else {
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const float mean = RMS ? 0.f : warp_sum(s) / (float)D;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < D) {
      const float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, d = v[i].w - mean;
      sq += (a * a + b * b) + (cc * cc + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)D + eps);
  if (lane == 0) {
    if (!RMS && mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
  const long long orow = map_row(row, rpg, gstride, goff);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < D) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
      float o0, o1, o2, o3;
      if constexpr (RMS) {
        o0 = (v[i].x * rstd) * g.x; o1 = (v[i].y * rstd) * g.y; o2 = (v[i].z * rstd) * g.z; o3 = (v[i].w * rstd) * g.w;
      } else {
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
        o0 = (v[i].x - mean) * rstd * g.x + b.x; o1 = (v[i].y - mean) * rstd * g.y + b.y;
        o2 = (v[i].z - mean) * rstd * g.z + b.z; o3 = (v[i].w - mean) * rstd * g.w + b.w;
      }
      if (y_is_f32) {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + orow * ldy + c) = make_float4(o0, o1, o2, o3);
      } else {
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + orow * ldy + c) =
            make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
      }
    }
  }
}

// Backward: a 256-thread block walks rows blockIdx.x, +gridDim.x, ...; thread t owns float4 column groups
// (g*256 + t)*4.  dgamma/dbeta partials stay in registers and are written once per block to the workspace.
constexpr int LNB_THREADS = 256;
constexpr int LNB_MAX_BLOCKS = 592;  // 148 SMs x 4 resident blocks

template <int G, bool RMS = false>
__global__ void __launch_bounds__(LNB_THREADS) ln_bwd_kernel(
    const void* __restrict__ dy, int dy_is_f32, long long lddy, int rpg, int gstride, int goff,
    const float* __restrict__ x, long long ldx, const float* __restrict__ gamma, const float* __restrict__ mean,
    const float* __restrict__ rstd, int rows, int D, float* __restrict__ dx, long long lddx,
    const float* __restrict__ dx_add, long long ldadd, float* __restrict__ part) {
  __shared__ float s_red[2][8][2];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  float4 gm[G], dg[G], db[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const int c = (g * LNB_THREADS + t) * 4;
    gm[g] = c < D ? __ldg(reinterpret_cast<const float4*>(gamma + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    dg[g] = make_float4(0.f, 0.f, 0.f, 0.f);
    db[g] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invD = 1.0f / (float)D;
  int par = 0;
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    const float mu = RMS ? 0.f : mean[r], rs = rstd[r];
    const long long yr = map_row(r, rpg, gstride, goff);
    float4 xh[G], dyv[G];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int c = (g * LNB_THREADS + t) * 4;
      if (c < D) {
        const float4 xv = *reinterpret_cast<const float4*>(x + (long long)r * ldx + c);
        if (dy_is_f32) {
          dyv[g] = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) + yr * lddy + c);
        } else {
          const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(dy) + yr * lddy + c);
          dyv[g] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
        }
        xh[g] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
        const float a0 = dyv[g].x * gm[g].x, a1 = dyv[g].y * gm[g].y, a2 = dyv[g].z * gm[g].z, a3 = dyv[g].w * gm[g].w;
        s1 += (a0 + a1) + (a2 + a3);
        s2 += (a0 * xh[g].x + a1 * xh[g].y) + (a2 * xh[g].z + a3 * xh[g].w);
      } else {
        xh[g] = make_float4(0.f, 0.f, 0.f, 0.f);
        dyv[g] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if constexpr (RMS) s1 = 0.f;   // no centring: the mean(dy * gamma) term drops out
    s1 = warp_sum(s1); s2 = warp_sum(s2);
    if (lane == 0) { s_red[par][warp][0] = s1; s_red[par][warp][1] = s2; }
    __syncthreads();
    s1 = 0.f; s2 = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { s1 += s_red[par][w][0]; s2 += s_red[par][w][1]; }
    par ^= 1;
    const float m1 = s1 * invD, m2 = s2 * invD;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int c = (g * LNB_THREADS + t) * 4;
      if (c < D) {
        float4 o;
        o.x = rs * (dyv[g].x * gm[g].x - m1 - xh[g].x * m2);
        o.y = rs * (dyv[g].y * gm[g].y - m1 - xh[g].y * m2);
        o.z = rs * (dyv[g].z * gm[g].z - m1 - xh[g].z * m2);
        o.w = rs * (dyv[g].w * gm[g].w - m1 - xh[g].w * m2);
        if (dx_add) {
          const float4 a = *reinterpret_cast<const float4*>(dx_add + (long long)r * ldadd + c);
          o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w;
        }
        if (dx) *reinterpret_cast<float4*>(dx + (long long)r * lddx + c) = o;
        dg[g].x += dyv[g].x * xh[g].x; dg[g].y += dyv[g].y * xh[g].y; dg[g].z += dyv[g].z * xh[g].z; dg[g].w += dyv[g].w * xh[g].w;
        db[g].x += dyv[g].x; db[g].y += dyv[g].y; db[g].z += dyv[g].z; db[g].w += dyv[g].w;
      }
    }
  }
  if (part == nullptr) return;   // frozen LayerNorm (the LM's own norms): only dx is wanted
  float* pg = part + (long long)blockIdx.x * 2 * D;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const int c = (g * LNB_THREADS + t) * 4;
    if (c < D) {
      *reinterpret_cast<float4*>(pg + c) = dg[g];
      *reinterpret_cast<float4*>(pg + D + c) = db[g];
    }
  }
}

// Column-sum of the per-block partials: 64 columns x 4 row groups per 256-thread block (coalesced 256-byte row
// segments), the partial rows split over gridDim.y chunks so ~500 blocks share the 2 * D * nblocks floats (a
// 64-block grid left more than half of the SMs idle and took as long as the backward kernel's own tail);
// chunk results are combined with one red.global.add per column (dgamma / dbeta accumulate anyway).
constexpr int LNR_CHUNKS = 8;
__global__ void __launch_bounds__(256) ln_bwd_reduce_kernel(const float* __restrict__ part, int nblocks, int D,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float s_acc[4][64];
  const int c = blockIdx.x * 64 + (threadIdx.x & 63);  // over 2*D
  const int rg = threadIdx.x >> 6;
  const int per = (nblocks + gridDim.y - 1) / gridDim.y;
  const int b0 = blockIdx.y * per, b1 = min(nblocks, b0 + per);
  float s0 = 0.f, s1 = 0.f;
  if (c < 2 * D) {
    int b = b0 + rg;
    for (; b + 4 < b1; b += 8) {
      s0 += part[(long long)b * 2 * D + c];
      s1 += part[(long long)(b + 4) * 2 * D + c];
    }
    if (b < b1) s0 += part[(long long)b * 2 * D + c];
  }
  s_acc[rg][threadIdx.x & 63] = s0 + s1;
  __syncthreads();
  if (rg == 0 && c < 2 * D) {
    const float s = (s_acc[0][threadIdx.x] + s_acc[1][threadIdx.x]) + (s_acc[2][threadIdx.x] + s_acc[3][threadIdx.x]);
    if (c < D) { if (dgamma) atomicAdd(dgamma + c, s); }
    else if (dbeta) atomicAdd(dbeta + (c - D), s);
  }
}

}  // namespace ofk

extern "C" int ofk_layernorm_fwd(const float* x, long long ldx, const float* gamma, const float* beta, float eps,
                                 int rows, int D, void* y, int y_is_f32, long long ldy, int rows_per_group,
                                 int group_stride, int group_offset, float* mean, float* rstd, void* stream_) {
  using namespace ofk;
  if (!x || !gamma || !beta || !y) return ofk_set_error(OFK_ERR_ARG, "layernorm: null pointer");
  if (rows <= 0) return 0;
  if (D <= 0 || D % 4 != 0 || D > 4096) return ofk_set_error(OFK_ERR_ARG, "layernorm: D must be a multiple of 4, <= 4096");
  if (ldx % 4 != 0 || ldy % 4 != 0) return ofk_set_error(OFK_ERR_ALIGN, "layernorm: row strides must be multiples of 4");
  cudaStream_t s = (cudaStream_t)stream_;
  const int grid = (rows + 3) / 4;
  if (D <= 1024)
    ln_fwd_kernel<8><<<grid, 128, 0, s>>>(x, ldx, gamma, beta, eps, rows, D, y, y_is_f32, ldy, rows_per_group, group_stride, group_offset, mean, rstd);
  else if (D <= 2048)
    ln_fwd_kernel<16><<<grid, 128, 0, s>>>(x, ldx, gamma, beta, eps, rows, D, y, y_is_f32, ldy, rows_per_group, group_stride, group_offset, mean, rstd);
  else
    ln_fwd_kernel<32><<<grid, 128, 0, s>>>(x, ldx, gamma, beta, eps, rows, D, y, y_is_f32, ldy, rows_per_group, group_stride, group_offset, mean, rstd);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" long long ofk_layernorm_bwd_workspace(int rows, int D) {
  (void)rows;
  return (long long)ofk::LNB_MAX_BLOCKS * 2 * D * sizeof(float);
}

extern "C" int ofk_layernorm_bwd(const void* dy, int dy_is_f32, long long lddy, int rows_per_group, int group_stride,
                                 int group_offset, const float* x, long long ldx, const float* gamma, const float* mean,
                                 const float* rstd, int rows, int D, float* dx, long long lddx, const float* dx_add,
                                 long long ldadd, float* dgamma, float* dbeta, void* workspace, void* stream_) {
  using namespace ofk;
  if (!dy || !x || !gamma || !mean || !rstd || !workspace) return ofk_set_error(OFK_ERR_ARG, "layernorm bwd: null pointer");
  if (!dx && !dgamma && !dbeta) return 0;
  if (rows <= 0) return 0;
  if (D <= 0 || D % 4 != 0 || D > 4096) return ofk_set_error(OFK_ERR_ARG, "layernorm bwd: D must be a multiple of 4, <= 4096");
  if (ldx % 4 != 0 || lddy % 4 != 0 || lddx % 4 != 0 || (dx_add && ldadd % 4 != 0))
    return ofk_set_error(OFK_ERR_ALIGN, "layernorm bwd: row strides must be multiples of 4");
  cudaStream_t s = (cudaStream_t)stream_;
  const int nblocks = rows < LNB_MAX_BLOCKS ? rows : LNB_MAX_BLOCKS;
  float* part = (dgamma || dbeta) ? reinterpret_cast<float*>(workspace) : nullptr;
  if (D <= 1024)
    ln_bwd_kernel<1><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, rows_per_group, group_stride, group_offset, x, ldx, gamma, mean, rstd, rows, D, dx, lddx, dx_add, ldadd, part);
  else if (D <= 2048)
    ln_bwd_kernel<2><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, rows_per_group, group_stride, group_offset, x, ldx, gamma, mean, rstd, rows, D, dx, lddx, dx_add, ldadd, part);
  else
    ln_bwd_kernel<4><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, rows_per_group, group_stride, group_offset, x, ldx, gamma, mean, rstd, rows, D, dx, lddx, dx_add, ldadd, part);
  OFK_CHECK_LAUNCH();
  if (dgamma || dbeta) {
    ln_bwd_reduce_kernel<<<dim3((2 * D + 63) / 64, nblocks >= 64 ? LNR_CHUNKS : 1), 256, 0, s>>>(part, nblocks, D, dgamma, dbeta);
    OFK_CHECK_LAUNCH();
  }
  return 0;
}

extern "C" int ofk_rmsnorm_fwd(const float* x, long long ldx, const float* gamma, float eps, int rows, int D, void* y,
                               long long ldy, float* rstd, void* stream_) {
  using namespace ofk;
  if (!x || !gamma || !y) return ofk_set_error(OFK_ERR_ARG, "rmsnorm: null pointer");
  if (rows <= 0) return 0;
  if (D <= 0 || D % 4 != 0 || D > 4096) return ofk_set_error(OFK_ERR_ARG, "rmsnorm: D must be a multiple of 4, <= 4096");
  if (ldx % 4 != 0 || ldy % 4 != 0) return ofk_set_error(OFK_ERR_ALIGN, "rmsnorm: row strides must be multiples of 4");
  cudaStream_t s = (cudaStream_t)stream_;
  const int grid = (rows + 3) / 4;
  if (D <= 1024)
    ln_fwd_kernel<8, true><<<grid, 128, 0, s>>>(x, ldx, gamma, nullptr, eps, rows, D, y, 0, ldy, 0, 0, 0, nullptr, rstd);
  else if (D <= 2048)
    ln_fwd_kernel<16, true><<<grid, 128, 0, s>>>(x, ldx, gamma, nullptr, eps, rows, D, y, 0, ldy, 0, 0, 0, nullptr, rstd);
  else
    ln_fwd_kernel<32, true><<<grid, 128, 0, s>>>(x, ldx, gamma, nullptr, eps, rows, D, y, 0, ldy, 0, 0, 0, nullptr, rstd);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_rmsnorm_bwd(const void* dy, int dy_is_f32, long long lddy, const float* x, long long ldx,
                               const float* gamma, const float* rstd, int rows, int D, float* dx, long long lddx,
                               const float* dx_add, long long ldadd, void* stream_) {
  using namespace ofk;
  if (!dy || !x || !gamma || !rstd || !dx) return ofk_set_error(OFK_ERR_ARG, "rmsnorm bwd: null pointer");
  if (rows <= 0) return 0;
  if (D <= 0 || D % 4 != 0 || D > 4096) return ofk_set_error(OFK_ERR_ARG, "rmsnorm bwd: D must be a multiple of 4, <= 4096");
  if (ldx % 4 != 0 || lddy % 4 != 0 || lddx % 4 != 0 || (dx_add && ldadd % 4 != 0))
    return ofk_set_error(OFK_ERR_ALIGN, "rmsnorm bwd: row strides must be multiples of 4");
  cudaStream_t s = (cudaStream_t)stream_;
  const int nblocks = rows < LNB_MAX_BLOCKS ? rows : LNB_MAX_BLOCKS;
  if (D <= 1024)
    ln_bwd_kernel<1, true><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, 0, 0, 0, x, ldx, gamma, nullptr, rstd, rows, D, dx, lddx, dx_add, ldadd, nullptr);
  else if (D <= 2048)
    ln_bwd_kernel<2, true><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, 0, 0, 0, x, ldx, gamma, nullptr, rstd, rows, D, dx, lddx, dx_add, ldadd, nullptr);
  else
    ln_bwd_kernel<4, true><<<nblocks, LNB_THREADS, 0, s>>>(dy, dy_is_f32, lddy, 0, 0, 0, x, ldx, gamma, nullptr, rstd, rows, D, dx, lddx, dx_add, ldadd, nullptr);
  OFK_CHECK_LAUNCH();
  return 0;
}
