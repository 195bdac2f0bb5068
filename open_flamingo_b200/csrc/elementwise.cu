// Small HBM-bound kernels around the GEMMs: mask prefix-sum, casts, gate backward, ViT patch gather,
// fused AdamW.  All are vectorised (16-byte accesses), grid-stride, one pass over their data.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ofk_internal.h"
#include "ofk_ptx.cuh"

namespace ofk {

static inline int grid_for(long long work_items, int threads) {
  long long b = (work_items + threads - 1) / threads;
  const long long cap = 148LL * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ---- text_time (helpers.py:199-208): one warp per batch row, ballot-based inclusive scan.
__global__ void text_time_kernel(const long long* __restrict__ ids, long long media_id, int t_txt, int n_loc,
                                 const unsigned char* __restrict__ loc, int cached, int* __restrict__ out) {
  const int b = blockIdx.x, lane = threadIdx.x;
  if (cached) {
    int cnt = 0;
    for (int i = lane; i < n_loc; i += 32) cnt += loc[(long long)b * n_loc + i] ? 1 : 0;
    cnt = (int)warp_sum((float)cnt);  // n_loc is far below 2^24: exact
    for (int i = lane; i < t_txt; i += 32) out[(long long)b * t_txt + i] = cnt;
    return;
  }
  int running = 0;
  for (int base = 0; base < t_txt; base += 32) {
    const int i = base + lane;
    bool flag = false;
    if (i < t_txt) flag = loc ? (loc[(long long)b * n_loc + i] != 0) : (ids[(long long)b * t_txt + i] == media_id);
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    const int incl = running + __popc(m & (0xffffffffu >> (31 - lane)));
    if (i < t_txt) out[(long long)b * t_txt + i] = incl;
    running += __popc(m);
  }
}

// ---- training labels (train_utils.py:102-106 LAION, :126-149 MMC4) ------------------------------------------
// labels = input_ids with pad and <image> masked to -100; interleaved (MMC4) rows additionally mask every token
// before the first <image> and every token between an <|endofchunk|> and the next <image> (the <|endofchunk|>
// itself keeps its label).  The reference walks each row with Python while-loops; here it is a two-state scan
// ("open" after an <image>, "closed" after an <|endofchunk|>, closed initially): 256 tokens per pass, coalesced,
// the state a token sees = the kind of the latest <image>/<|endofchunk|> strictly before it (ballot + clz inside a
// warp, 8 warp summaries in shared memory, a block-uniform carry between passes).
__global__ void __launch_bounds__(256) make_labels_kernel(const long long* __restrict__ ids, long long ld_ids, int T,
                                                          long long pad_id, long long media_id, long long eoc_id,
                                                          int interleaved, long long* __restrict__ labels,
                                                          long long ld_lab) {
  __shared__ int s_last[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long* src = ids + (long long)blockIdx.x * ld_ids;
  long long* dst = labels + (long long)blockIdx.x * ld_lab;
  int carry = 0;   // 1 = open: the latest marker so far was an <image>
  for (int t0 = 0; t0 < T; t0 += 256) {
    const int t = t0 + tid;
    const long long id = t < T ? src[t] : pad_id;
    // the reference compares against the labels AFTER pad masking (train_utils.py:127-128), so a marker id that
    // coincides with the pad id is never seen as a marker
    int kind = 0;
    if (t < T && id != pad_id) kind = (id == media_id) ? 1 : ((id == eoc_id) ? 2 : 0);
    const unsigned nz = __ballot_sync(0xffffffffu, kind != 0);
    const unsigned below = nz & ((1u << lane) - 1u);
    const int prev = __shfl_sync(0xffffffffu, kind, below ? 31 - __clz(below) : 0);
    int st = below ? prev : 0;                                   // 0 = no marker earlier in this warp
    if (lane == 31) s_last[warp] = kind != 0 ? kind : st;        // latest marker of the whole warp
    __syncthreads();
    for (int w = warp - 1; w >= 0 && st == 0; --w) st = s_last[w];
    int tile_last = 0;
    for (int w = 7; w >= 0 && tile_last == 0; --w) tile_last = s_last[w];
    const bool open = st == 0 ? (carry != 0) : (st == 1);
    if (t < T) {
      const bool masked = id == pad_id || id == media_id || (interleaved && !open);
      dst[t] = masked ? -100LL : id;
    }
    if (tile_last != 0) carry = tile_last == 1;
    __syncthreads();
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  const long long n8 = n / 8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = reinterpret_cast<const float4*>(src)[2 * i], b = reinterpret_cast<const float4*>(src)[2 * i + 1];
    reinterpret_cast<uint4*>(dst)[i] = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
  }
  for (long long i = n8 * 8 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __float2bfloat16_rn(src[i]);
}

// ---- gate backward: dbranch = dout * tanh(g) (bf16); dgate += (1 - tanh(g)^2) * <dout, branch>
__global__ void __launch_bounds__(256) gate_bwd_kernel(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ branch,
                                                       const float* __restrict__ gate, __nv_bfloat16* __restrict__ dbranch,
                                                       float* __restrict__ dgate, long long n) {
  __shared__ float s_part[8];
  const float tg = gate ? tanhf(__ldg(gate)) : 1.0f;
  const long long n8 = n / 8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = reinterpret_cast<const float4*>(dout)[2 * i], b = reinterpret_cast<const float4*>(dout)[2 * i + 1];
    if (gate) {
      const uint4 br = reinterpret_cast<const uint4*>(branch)[i];
      acc += a.x * bf16_lo(br.x) + a.y * bf16_hi(br.x) + a.z * bf16_lo(br.y) + a.w * bf16_hi(br.y) +
             b.x * bf16_lo(br.z) + b.y * bf16_hi(br.z) + b.z * bf16_lo(br.w) + b.w * bf16_hi(br.w);
    }
    reinterpret_cast<uint4*>(dbranch)[i] = make_uint4(pack_bf16x2(a.x * tg, a.y * tg), pack_bf16x2(a.z * tg, a.w * tg),
                                                      pack_bf16x2(b.x * tg, b.y * tg), pack_bf16x2(b.z * tg, b.w * tg));
  }
  if (gate && dgate) {
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += s_part[w];
      atomicAdd(dgate, s * (1.0f - tg * tg));
    }
  }
}

// ---- rotary position embedding (HF apply_rotary_pos_emb), in place on the q / k heads of fused bf16 rows.
// One thread per (row, head, 8-column chunk of the head's first half): it owns columns i and i + hd/2, the pair
// rotate_half mixes.  __fmul_rn / __fadd_rn keep the products and the sum separately rounded, as torch computes them.
__device__ __forceinline__ void load8f(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void unpack8(uint4 u, float (&v)[8]) {
  v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y);
  v[4] = bf16_lo(u.z); v[5] = bf16_hi(u.z); v[6] = bf16_lo(u.w); v[7] = bf16_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

__global__ void __launch_bounds__(256) rope_kernel(__nv_bfloat16* __restrict__ x, long long ldx, int T, int nheads, int hd,
                                                   const float* __restrict__ cosp, const float* __restrict__ sinp,
                                                   long long csb, int inverse, long long total) {
  const int chunks = hd / 16;
  const int half = hd / 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const int c = (int)(idx % chunks);
    const long long rh = idx / chunks;
    const int h = (int)(rh % nheads);
    const long long r = rh / nheads;
    const long long b = r / T, t = r % T;
    const int i0 = c * 8;
    __nv_bfloat16* p = x + r * ldx + (long long)h * hd + i0;
    const float* cs = cosp + b * csb + t * hd + i0;
    const float* sn = sinp + b * csb + t * hd + i0;
    float lo[8], hi[8], cl[8], ch[8], sl[8], sh[8];
    unpack8(*reinterpret_cast<const uint4*>(p), lo);
    unpack8(*reinterpret_cast<const uint4*>(p + half), hi);
    load8f(cs, cl); load8f(cs + half, ch); load8f(sn, sl); load8f(sn + half, sh);
    float olo[8], ohi[8];
    if (!inverse) {
      // out = x * cos + rotate_half(x) * sin,  rotate_half(x) = (-x_hi, x_lo)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        olo[i] = __fsub_rn(__fmul_rn(lo[i], cl[i]), __fmul_rn(hi[i], sl[i]));
        ohi[i] = __fadd_rn(__fmul_rn(hi[i], ch[i]), __fmul_rn(lo[i], sh[i]));
      }
    } else {
      // autograd: dx = bf16(d * cos) + rotate_half^T(bf16(d * sin)),  rotate_half^T(y) = (y_hi, -y_lo)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        olo[i] = bf16_round(lo[i] * cl[i]) + bf16_round(hi[i] * sh[i]);
        ohi[i] = bf16_round(hi[i] * ch[i]) - bf16_round(lo[i] * sl[i]);
      }
    }
    *reinterpret_cast<uint4*>(p) = pack8(olo);
    *reinterpret_cast<uint4*>(p + half) = pack8(ohi);
  }
}

// ---- SwiGLU backward on the packed [g | u] layout (OFK_SWIGLU_GROUP): one thread per 8 h columns of one row.
__global__ void __launch_bounds__(256) swiglu_bwd_kernel(const __nv_bfloat16* __restrict__ dh, long long lddh,
                                                         const __nv_bfloat16* __restrict__ gu, long long ldgu, int I,
                                                         __nv_bfloat16* __restrict__ dgu, long long lddgu, long long total) {
  const int per_row = I / 8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const long long r = idx / per_row;
    const int j8 = (int)(idx % per_row) * 8;                               // first h column
    const int pc = (j8 / OFK_SWIGLU_GROUP) * 2 * OFK_SWIGLU_GROUP + j8 % OFK_SWIGLU_GROUP;   // its gate column
    float d[8], g[8], u[8], dg[8], du[8];
    unpack8(*reinterpret_cast<const uint4*>(dh + r * lddh + j8), d);
    unpack8(*reinterpret_cast<const uint4*>(gu + r * ldgu + pc), g);
    unpack8(*reinterpret_cast<const uint4*>(gu + r * ldgu + pc + OFK_SWIGLU_GROUP), u);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      du[i] = d[i] * bf16_round(silu(g[i]));
      dg[i] = bf16_round(d[i] * u[i]) * silu_grad(g[i]);
    }
    *reinterpret_cast<uint4*>(dgu + r * lddgu + pc) = pack8(dg);
    *reinterpret_cast<uint4*>(dgu + r * lddgu + pc + OFK_SWIGLU_GROUP) = pack8(du);
  }
}

__global__ void add_f32_kernel(float* __restrict__ dst, const float* __restrict__ src, long long n) {
  const long long n4 = n / 4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 a = reinterpret_cast<float4*>(dst)[i];
    const float4 b = reinterpret_cast<const float4*>(src)[i];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(dst)[i] = a;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] += src[i];
}

// ---- ViT patch gather: one thread per (patch, channel, patch-row); writes P contiguous bf16.
__global__ void patchify_kernel(const float* __restrict__ img, int n, int H, int W, int P, __nv_bfloat16* __restrict__ out,
                                long long ldp) {
  const int gh = H / P, gw = W / P;
  const long long total = (long long)n * gh * gw * 3 * P;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const int ph = (int)(idx % P);
    long long r = idx / P;
    const int c = (int)(r % 3); r /= 3;
    const int px = (int)(r % gw); r /= gw;
    const int py = (int)(r % gh);
    const int im = (int)(r / gh);
    const float* src = img + (((long long)im * 3 + c) * H + (py * P + ph)) * W + px * P;
    __nv_bfloat16* dst = out + ((long long)(im * gh + py) * gw + px) * ldp + (c * P + ph) * P;
    for (int pw = 0; pw < P; ++pw) dst[pw] = __float2bfloat16_rn(src[pw]);
  }
}
// zero the padding columns [kvalid, ldp)
__global__ void patch_pad_kernel(__nv_bfloat16* __restrict__ out, long long rows, int kvalid, long long ldp) {
  const int pad = (int)(ldp - kvalid);
  const long long total = rows * pad;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride)
    out[(idx / pad) * ldp + kvalid + (idx % pad)] = __float2bfloat16_rn(0.f);
}

__global__ void vit_assemble_kernel(const __nv_bfloat16* __restrict__ pe, const float* __restrict__ cls,
                                    const float* __restrict__ pos, int n, int g, int D, float* __restrict__ tok) {
  const long long total = (long long)n * (g + 1) * (D / 4);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const int c = (int)(idx % (D / 4)) * 4;
    const long long r = idx / (D / 4);
    const int tkn = (int)(r % (g + 1));
    const long long im = r / (g + 1);
    float4 v;
    if (tkn == 0) {
      v = *reinterpret_cast<const float4*>(cls + c);
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(pe + (im * g + (tkn - 1)) * D + c);
      v = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
    const float4 p = *reinterpret_cast<const float4*>(pos + (long long)tkn * D + c);
    v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    *reinterpret_cast<float4*>(tok + r * D + c) = v;
  }
}

// ---- fused AdamW (decoupled weight decay, torch.optim.AdamW semantics) + bf16 operand refresh
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, __nv_bfloat16* __restrict__ w16, long long n, float lr, float b1,
                             float b2, float eps, float wd, float bc1, float bc2, const float* __restrict__ clip,
                             const float* __restrict__ step_dev, const float* __restrict__ lr_dev) {
  const float cs = clip ? __ldg(clip) : 1.0f;
  if (step_dev) {  // device-resident step counter (CUDA-graph replays cannot bake the bias corrections in)
    const float st = __ldg(step_dev);
    bc1 = 1.0f - powf(b1, st);
    bc2 = 1.0f - powf(b2, st);
  }
  if (lr_dev) lr = __ldg(lr_dev);
  const float step = lr / bc1;
  const float inv_sqrt_bc2 = rsqrtf(bc2);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gi = g[i] * cs;
    float pi = p[i];
    pi *= (1.0f - lr * wd);
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    pi -= step * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
    p[i] = pi;
    if (w16) w16[i] = __float2bfloat16_rn(pi);
  }
}

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  __shared__ float s_part[8];
  const long long stride = (long long)gridDim.x * blockDim.x;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc += x[i] * x[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += s_part[w];
    atomicAdd(out, s);
  }
}

}  // namespace ofk

using namespace ofk;

extern "C" int ofk_text_time(const long long* input_ids, long long media_token_id, int batch, int t_txt, int n_loc,
                             const unsigned char* media_locations, int use_cached_media, int* text_time, void* stream) {
  if (!text_time || (!input_ids && !media_locations)) return ofk_set_error(OFK_ERR_ARG, "text_time: null pointer");
  if (use_cached_media && !media_locations) return ofk_set_error(OFK_ERR_ARG, "text_time: cached mode needs media_locations");
  if (!use_cached_media && media_locations && n_loc != t_txt)
    return ofk_set_error(OFK_ERR_ARG, "text_time: media_locations length must equal t_txt (helpers.py:175-178)");
  if (batch <= 0 || t_txt <= 0) return 0;
  text_time_kernel<<<batch, 32, 0, (cudaStream_t)stream>>>(input_ids, media_token_id, t_txt, n_loc, media_locations,
                                                           use_cached_media, text_time);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_make_labels(const long long* input_ids, long long ld_ids, int batch, int t_txt, long long pad_token_id,
                               long long media_token_id, long long endofchunk_token_id, int interleaved,
                               long long* labels, long long ld_labels, void* stream) {
  if (batch <= 0 || t_txt <= 0) return 0;
  if (!input_ids || !labels) return ofk_set_error(OFK_ERR_ARG, "make_labels: null pointer");
  if (ld_ids < t_txt || ld_labels < t_txt) return ofk_set_error(OFK_ERR_ARG, "make_labels: row stride shorter than the row");
  make_labels_kernel<<<batch, 256, 0, (cudaStream_t)stream>>>(input_ids, ld_ids, t_txt, pad_token_id, media_token_id,
                                                              endofchunk_token_id, interleaved, labels, ld_labels);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_cast_f32_bf16(const float* src, void* dst, long long n, void* stream) {
  if (!src || !dst) return ofk_set_error(OFK_ERR_ARG, "cast: null pointer");
  if (n <= 0) return 0;
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 15))
    return ofk_set_error(OFK_ERR_ALIGN, "cast: pointers must be 16-byte aligned");
  cast_f32_bf16_kernel<<<grid_for(n / 8 + 1, 256), 256, 0, (cudaStream_t)stream>>>(src, (__nv_bfloat16*)dst, n);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_gate_bwd(const float* dout, const void* branch, const float* gate, void* dbranch, float* dgate,
                            long long n, void* stream) {
  if (!dout || !dbranch || (gate && !branch)) return ofk_set_error(OFK_ERR_ARG, "gate_bwd: null pointer");
  if (n <= 0) return 0;
  if (n % 8 != 0) return ofk_set_error(OFK_ERR_ARG, "gate_bwd: n must be a multiple of 8");
  gate_bwd_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(dout, (const __nv_bfloat16*)branch, gate,
                                                                           (__nv_bfloat16*)dbranch, dgate, n);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_rope(void* x, long long ldx, int batch, int T, int nheads, int head_dim, const float* cos,
                        const float* sin, long long cs_bstride, int inverse, void* stream) {
  if (!x || !cos || !sin) return ofk_set_error(OFK_ERR_ARG, "rope: null pointer");
  if (batch <= 0 || T <= 0 || nheads <= 0) return 0;
  if (head_dim <= 0 || head_dim % 16 != 0 || ldx < (long long)nheads * head_dim)
    return ofk_set_error(OFK_ERR_ARG, "rope: head_dim must be a multiple of 16 and the heads must fit the row");
  if ((reinterpret_cast<uintptr_t>(x) & 15) || ldx % 8 != 0 || (reinterpret_cast<uintptr_t>(cos) & 15) ||
      (reinterpret_cast<uintptr_t>(sin) & 15) || cs_bstride % 4 != 0)
    return ofk_set_error(OFK_ERR_ALIGN, "rope: x / cos / sin must be 16-byte aligned with 16-byte row strides");
  const long long total = (long long)batch * T * nheads * (head_dim / 16);
  rope_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)x, ldx, T, nheads, head_dim, cos,
                                                                      sin, cs_bstride, inverse, total);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_swiglu_bwd(const void* dh, long long lddh, const void* gu, long long ldgu, int rows, int I, void* dgu,
                              long long lddgu, void* stream) {
  if (!dh || !gu || !dgu) return ofk_set_error(OFK_ERR_ARG, "swiglu_bwd: null pointer");
  if (rows <= 0) return 0;
  if (I <= 0 || I % OFK_SWIGLU_GROUP != 0) return ofk_set_error(OFK_ERR_ARG, "swiglu_bwd: I must be a multiple of 16");
  if ((reinterpret_cast<uintptr_t>(dh) & 15) || (reinterpret_cast<uintptr_t>(gu) & 15) ||
      (reinterpret_cast<uintptr_t>(dgu) & 15) || lddh % 8 != 0 || ldgu % 8 != 0 || lddgu % 8 != 0)
    return ofk_set_error(OFK_ERR_ALIGN, "swiglu_bwd: operands must be 16-byte aligned with 16-byte row strides");
  const long long total = (long long)rows * (I / 8);
  swiglu_bwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)dh, lddh, (const __nv_bfloat16*)gu, ldgu, I, (__nv_bfloat16*)dgu, lddgu, total);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_add_f32(float* dst, const float* src, long long n, void* stream) {
  if (!dst || !src) return ofk_set_error(OFK_ERR_ARG, "add: null pointer");
  if (n <= 0) return 0;
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 15))
    return ofk_set_error(OFK_ERR_ALIGN, "add: pointers must be 16-byte aligned");
  add_f32_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream>>>(dst, src, n);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_patchify(const float* images, int n, int H, int W, int P, void* patches, long long ldp, void* stream) {
  if (!images || !patches) return ofk_set_error(OFK_ERR_ARG, "patchify: null pointer");
  if (n <= 0) return 0;
  if (P <= 0 || H % P || W % P || ldp < 3LL * P * P) return ofk_set_error(OFK_ERR_ARG, "patchify: bad geometry");
  const long long rows = (long long)n * (H / P) * (W / P);
  patchify_kernel<<<grid_for(rows * 3 * P, 256), 256, 0, (cudaStream_t)stream>>>(images, n, H, W, P, (__nv_bfloat16*)patches, ldp);
  OFK_CHECK_LAUNCH();
  if (ldp > 3LL * P * P) {
    patch_pad_kernel<<<grid_for(rows * (ldp - 3 * P * P), 256), 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)patches, rows, 3 * P * P, ldp);
    OFK_CHECK_LAUNCH();
  }
  return 0;
}

extern "C" int ofk_vit_assemble(const void* patch_emb, const float* class_emb, const float* pos_emb, int n, int g, int D,
                                float* tokens, void* stream) {
  if (!patch_emb || !class_emb || !pos_emb || !tokens) return ofk_set_error(OFK_ERR_ARG, "vit_assemble: null pointer");
  if (n <= 0) return 0;
  if (D % 4 != 0) return ofk_set_error(OFK_ERR_ARG, "vit_assemble: D must be a multiple of 4");
  vit_assemble_kernel<<<grid_for((long long)n * (g + 1) * (D / 4), 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)patch_emb, class_emb, pos_emb, n, g, D, tokens);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_adamw(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, void* w_bf16, long long n,
                         float lr, float beta1, float beta2, float eps, float wd, float bias_corr1, float bias_corr2,
                         const float* clip_scale, const float* step_dev, const float* lr_dev, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq) return ofk_set_error(OFK_ERR_ARG, "adamw: null pointer");
  if (n <= 0) return 0;
  adamw_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, (__nv_bfloat16*)w_bf16, n,
                                                                    lr, beta1, beta2, eps, wd, bias_corr1, bias_corr2, clip_scale,
                                                                    step_dev, lr_dev);
  OFK_CHECK_LAUNCH();
  return 0;
}

extern "C" int ofk_sumsq(const float* x, long long n, float* out, void* stream) {
  if (!x || !out) return ofk_set_error(OFK_ERR_ARG, "sumsq: null pointer");
  if (n <= 0) return 0;
  sumsq_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, n, out);
  OFK_CHECK_LAUNCH();
  return 0;
}
