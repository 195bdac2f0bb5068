// bf16 x bf16 -> fp32 GEMM for sm_100a: TMA-staged operands (128B swizzle), tcgen05.mma with the
// accumulator in TMEM (double buffered), warp-specialised persistent CTAs, fused epilogues.
//
//   out[m, n] = epilogue( sum_k A(m, k) * B(n, k) )
//
// Operand storage ("major"):
//   K-major  : X is [rows, K] row-major (K contiguous)             -- forward  Y = X W^T
//   MN-major : X is [K, rows] row-major (rows contiguous)          -- dgrad (B = W) / wgrad (A = dY, B = X)
// so no transposed copies of weights or activations are ever materialised.
//
// This kernel replaces every nn.Linear on the reference hot path:
//   helpers.py:15-22 (FeedForward), :35-37 / :52-54 / :65 (PerceiverAttention to_q/to_kv/to_out),
//   :153-155 / :186-189 / :233 (MaskedCrossAttention to_q/to_kv/to_out), and the gate/residual
//   arithmetic of helpers.py:267-277 in its epilogue; plus the open_clip ViT linears (third party).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <mutex>
#include <unordered_map>

#include "ofk_internal.h"
#include "ofk_ptx.cuh"

namespace ofk {

constexpr int BM = 128;       // UMMA_M (cta_group::1)
constexpr int BK = 64;        // one 128-byte swizzle atom of bf16
constexpr int UMMA_K = 16;    // fixed for 16-bit inputs
// Warp roles.  The SM's issue arbiter favours the highest warp ids (B300_MICROARCH.md, "hi-wid-first"), so the
// single-thread TMA producer and MMA issuer sit ABOVE the eight math-heavy epilogue warps: with them at warps 0/1
// an ncu capture showed the tensor pipe only 57-68 % active on the K=2048 GELU GEMMs (issuer starved by epilogue
// math); epilogue warps must satisfy warp % 4 == TMEM lane quarter, which warps 0..7 do.

constexpr int NUM_EPI_WARPS = 8;
constexpr int WARP_TMA = 8, WARP_MMA = 9, WARP_TMEM = 10;   // warp 11 idles
constexpr int NUM_THREADS = 12 * 32;
constexpr int GROUP_M = 8;        // tile rasterisation: GROUP_M m-tiles x all n-tiles are walked together (L2 reuse)

struct GemmParams {
  int M, N, K;
  int splits;        // split-K factor (>1 only with the atomic epilogue)
  int kb_per_split;  // k-blocks per split
  void* out;
  long long ldo;
  void* out2;
  long long ldo2;
  const void* aux;
  long long ldaux;
  const float* bias;
  const float* gate;
  int stream_out;    // 1: epilogue outputs use st.global.cs (evict-first) so they do not displace the operand panels in L2
  // Grouped row maps (0 = identity): logical row r -> (r / rpg) * gs + go + r % rpg.  `out_*` places the rows of `out`
  // inside a larger interleaved buffer (the media / latent halves of PerceiverAttention's cat((x, latents), -2),
  // helpers.py:53); `ak_*` does the same for the REDUCTION rows of an MN-major A operand (wgrad over one half).
  int out_rpg, out_gs, out_go;
  int ak_rpg, ak_gs, ak_go;
  // Tail split (2-CTA kernel, splits == 1): the tiles of the last, partially filled round of the persistent grid
  // are cut into `tail_s` k-slices that run on otherwise idle SM pairs.  Slices 0..tail_s-2 dump their fp32
  // accumulators into `tail_ws` (register order, coalesced) and bump a per-warp flag; the last slice waits for the
  // flags, adds the partials to its own accumulator and runs the normal fused epilogue.  tail_s == 0: off.
  int tail_first;    // first rasterised tile index of the tail round
  int tail_s;        // k-slices per tail tile (2..4)
  int tail_kps;      // k-blocks per slice
  float* tail_ws;    // [(rem * (tail_s - 1))][2 CTAs][8 warps][4 rounds][8][32 lanes][4] floats
  int* tail_flags;   // [rem][2 CTAs][8 warps]
};
__device__ __forceinline__ long long map_rows(long long r, int rpg, int gs, int go) {
  return rpg > 0 ? (r / rpg) * gs + go + r % rpg : r;
}

// Work item -> (m tile, n tile, k split).  Within a split, tiles are walked in groups of GROUP_M m-tiles by all
// n-tiles, m fastest, so the ~74-148 tiles in flight share GROUP_M row panels of A and ~10-18 column panels of B
// through L2 (an ncu capture of the plain m-fastest order showed 650 MB of DRAM reads for 234 MB of operands).
__device__ __forceinline__ void work_to_tile(int w, int m_tiles, int n_tiles, int& mt, int& nt, int& ks) {
  const int per_split = m_tiles * n_tiles;
  ks = w / per_split;
  const int r = w - ks * per_split;
  const int group_sz = GROUP_M * n_tiles;
  const int g = r / group_sz;
  const int first_m = g * GROUP_M;
  const int gm = min(GROUP_M, m_tiles - first_m);
  const int in_g = r - g * group_sz;
  mt = first_m + in_g % gm;
  nt = in_g / gm;
}

// Work item of the 2-CTA kernel -> tile, k-block range and tail-split role (0 = whole tile, 1 = partial producer,
// 2 = owner of a split tile).
struct Work2 { int mt, nt, kb0, kb1, role, t, j; };
__device__ __forceinline__ Work2 decode_work2(const GemmParams& p, int w, int m_tiles, int n_tiles, int total_kb) {
  Work2 o;
  int ks;
  if (p.tail_s > 0 && w >= p.tail_first) {
    const int u = w - p.tail_first;
    o.t = u / p.tail_s;
    o.j = u - o.t * p.tail_s;
    work_to_tile(p.tail_first + o.t, m_tiles, n_tiles, o.mt, o.nt, ks);
    o.kb0 = o.j * p.tail_kps;
    o.kb1 = min(total_kb, o.kb0 + p.tail_kps);
    o.role = (o.j == p.tail_s - 1) ? 2 : 1;
  } else {
    work_to_tile(w, m_tiles, n_tiles, o.mt, o.nt, ks);
    o.kb0 = ks * p.kb_per_split;
    o.kb1 = min(total_kb, o.kb0 + p.kb_per_split);
    o.role = 0; o.t = 0; o.j = 0;
  }
  return o;
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_global_cg_v4(void* g, uint4 v) {
  asm volatile("st.global.cg.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(g), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_global_cg_v4(const void* g) {
  uint4 v;
  asm volatile("ld.global.cg.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(g) : "memory");
  return v;
}

template <int BN>
struct SmemLayout {
  static constexpr int A_BYTES = BM * BK * 2;   // 16 KiB
  static constexpr int B_BYTES = BN * BK * 2;   // 16/32 KiB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN == 256) ? 4 : 6;
  static constexpr int BAR_BYTES = 256;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + BAR_BYTES + NUM_EPI_WARPS * 32 * 128 + 1024;  // + epilogue staging + slack
};

// ----------------------------------------------------------------------------------------------
// Epilogue.  One warp drains 32 accumulator rows (lane = row) x 32 columns per round.  A lane owns a ROW, so a
// naive "each lane stores its row" epilogue issues warp stores that touch 32 different cache lines (an ncu capture
// showed the K=2048 GELU GEMMs pinned at 57-68 % tensor-pipe activity by exactly that L1 wavefront traffic).
// Instead every global access goes through a per-warp shared-memory staging tile and is re-issued TRANSPOSED:
// consecutive lanes touch consecutive 16-byte pieces of the same row (4 or 8 rows per instruction), i.e. full
// 64/128-byte segments.  The same staging tile is used for the epilogue's reads (residual, saved pre-activation).
constexpr int STAGE_ROW = 128;                     // unpadded 128 B rows; the 16-byte piece index is XOR-swizzled with
constexpr int STAGE_BYTES_PER_WARP = 32 * STAGE_ROW;   // (row & 7) so row-wise and piece-wise accesses are conflict-free
__device__ __forceinline__ uint32_t stage_off(int row, int piece) { return (uint32_t)(row * STAGE_ROW + ((piece ^ (row & 7)) << 4)); }


__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

// Store this warp's 32 x 32 tile (lane's row in `w`: WORDS = 32 for f32, 16 for bf16) to global, coalesced.
// MODE 0 = plain store, 1 = red.global.add.f32 (f32 only).
__device__ __forceinline__ void st_global_cs_v4(void* g, uint4 v) {
  asm volatile("st.global.cs.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(g), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int ELEM_BYTES, int MODE>
__device__ __forceinline__ void warp_store_tile(uint32_t stage, const uint32_t* w, void* gbase, long long ld, int row0,
                                                int col0, int M, int N, int streaming = 0, int rpg = 0, int gs = 0,
                                                int go = 0) {
  constexpr int PIECES = ELEM_BYTES * 2;            // 16-byte pieces per 32-element row: 8 (f32) or 4 (bf16)
  constexpr int EPP = 16 / ELEM_BYTES;              // elements per piece
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < PIECES; ++i)
    st_shared_v4(stage + stage_off(lane, i), make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]));
  __syncwarp();
  const int piece = lane % PIECES, rsub = lane / PIECES;
  const int col = col0 + piece * EPP;
#pragma unroll
  for (int it = 0; it < PIECES; ++it) {
    const int r = it * (32 / PIECES) + rsub;
    const uint4 v = ld_shared_v4(stage + stage_off(r, piece));
    const int row = row0 + r;
    if (row < M && col < N) {
      uint8_t* g = reinterpret_cast<uint8_t*>(gbase) + (map_rows(row, rpg, gs, go) * ld + col) * ELEM_BYTES;
      if constexpr (MODE == 0) {
        if (streaming) st_global_cs_v4(g, v);
        else *reinterpret_cast<uint4*>(g) = v;
      } else {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(g), "f"(__uint_as_float(v.x)),
                     "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w))
                     : "memory");
      }
    }
  }
  __syncwarp();
}

// Epilogue operand (residual / saved pre-activation) tile, two-phase so the global latency is hidden:
//   aux_prefetch: coalesced global loads of this warp's 32 x 32 tile into registers (issued one round ahead)
//   aux_commit  : registers -> staging tile -> each lane reads its own row
template <int ELEM_BYTES>
__device__ __forceinline__ void aux_prefetch(uint4 (&pre)[ELEM_BYTES * 2], const void* gbase, long long ld, int row0,
                                             int col0, int M, int N) {
  constexpr int PIECES = ELEM_BYTES * 2;
  constexpr int EPP = 16 / ELEM_BYTES;
  const int lane = threadIdx.x & 31;
  const int piece = lane % PIECES, rsub = lane / PIECES;
  const int col = col0 + piece * EPP;
#pragma unroll
  for (int it = 0; it < PIECES; ++it) {
    const int row = row0 + it * (32 / PIECES) + rsub;
    pre[it] = make_uint4(0u, 0u, 0u, 0u);
    if (row < M && col < N)
      pre[it] = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(gbase) + ((long long)row * ld + col) * ELEM_BYTES);
  }
}
template <int ELEM_BYTES>
__device__ __forceinline__ void aux_commit(uint32_t stage, const uint4 (&pre)[ELEM_BYTES * 2], uint32_t* w) {
  constexpr int PIECES = ELEM_BYTES * 2;
  const int lane = threadIdx.x & 31;
  const int piece = lane % PIECES, rsub = lane / PIECES;
#pragma unroll
  for (int it = 0; it < PIECES; ++it) st_shared_v4(stage + stage_off(it * (32 / PIECES) + rsub, piece), pre[it]);
  __syncwarp();
#pragma unroll
  for (int i = 0; i < PIECES; ++i) {
    const uint4 v = ld_shared_v4(stage + stage_off(lane, i));
    w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
  }
  __syncwarp();
}

// Store a 32-row x 16-column bf16 tile (lane's row in `w`) coalesced: two 16-byte pieces per row, 16 rows per
// instruction.  The SwiGLU epilogue's `h` output: one 32-column accumulator round yields 16 columns of h.
__device__ __forceinline__ void warp_store_tile16_bf16(uint32_t stage, const uint32_t (&w)[8], void* gbase, long long ld,
                                                       int row0, int col0, int M, int N, int streaming) {
  const int lane = threadIdx.x & 31;
  st_shared_v4(stage + stage_off(lane, 0), make_uint4(w[0], w[1], w[2], w[3]));
  st_shared_v4(stage + stage_off(lane, 1), make_uint4(w[4], w[5], w[6], w[7]));
  __syncwarp();
  const int piece = lane & 1, rsub = lane >> 1;
  const int col = col0 + piece * 8;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int r = it * 16 + rsub;
    const uint4 v = ld_shared_v4(stage + stage_off(r, piece));
    const int row = row0 + r;
    if (row < M && col < N) {
      void* g = reinterpret_cast<__nv_bfloat16*>(gbase) + (long long)row * ld + col;
      if (streaming) st_global_cs_v4(g, v);
      else *reinterpret_cast<uint4*>(g) = v;
    }
  }
  __syncwarp();
}

template <int EPI>
struct AuxBytes { static constexpr int value = (EPI == OFK_EPI_GATE_RESID_F32 || EPI == OFK_EPI_BIAS_RESID_F32) ? 4 : (EPI == OFK_EPI_DGELU_BF16 ? 2 : 0); };

__device__ __forceinline__ void pack32_bf16(const float (&v)[32], uint32_t (&w)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
}

// One round: rows [row0, row0+32) (lane = row) x columns [col0, col0+32), accumulators in `acc`.
template <int EPI>
__device__ __forceinline__ void epilogue32(const GemmParams& p, float gate_t, uint32_t stage, int row0, int col0,
                                           const uint32_t (&acc)[32], uint32_t* aux_row) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]);
  constexpr bool HAS_BIAS = EPI == OFK_EPI_BIAS_BF16 || EPI == OFK_EPI_BIAS_QGELU_BF16 || EPI == OFK_EPI_BIAS_GELU_BF16 ||
                            EPI == OFK_EPI_BIAS_RESID_F32;
  if constexpr (HAS_BIAS) {
    // every lane needs the same 32 bias values: broadcast loads (one wavefront each)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (col0 + 4 * i < p.N) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + i);
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    }
  }

  if constexpr (EPI == OFK_EPI_STORE_BF16 || EPI == OFK_EPI_BIAS_BF16 || EPI == OFK_EPI_BIAS_QGELU_BF16 ||
                EPI == OFK_EPI_BIAS_GELU_BF16) {
    if constexpr (EPI == OFK_EPI_BIAS_QGELU_BF16) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = quick_gelu(bf16_round(v[i]));
    }
    if constexpr (EPI == OFK_EPI_BIAS_GELU_BF16) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = gelu_exact(bf16_round(v[i]));
    }
    uint32_t w[16];
    pack32_bf16(v, w);
    warp_store_tile<2, 0>(stage, w, p.out, p.ldo, row0, col0, p.M, p.N, p.stream_out, p.out_rpg, p.out_gs, p.out_go);
  } else if constexpr (EPI == OFK_EPI_STORE_F32) {
    warp_store_tile<4, 0>(stage, acc, p.out, p.ldo, row0, col0, p.M, p.N, p.stream_out, p.out_rpg, p.out_gs, p.out_go);
  } else if constexpr (EPI == OFK_EPI_ATOMIC_F32) {
    warp_store_tile<4, 1>(stage, acc, p.out, p.ldo, row0, col0, p.M, p.N);
  } else if constexpr (EPI == OFK_EPI_GELU_DUAL) {
    // z = bf16(acc) is what the reference's Linear emits under autocast; GELU is taken of that.
    uint32_t wz[16], wh[16];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = bf16_round(v[i]);
    pack32_bf16(v, wz);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = gelu_exact(v[i]);
    pack32_bf16(v, wh);
    warp_store_tile<2, 0>(stage, wz, p.out, p.ldo, row0, col0, p.M, p.N, p.stream_out);
    warp_store_tile<2, 0>(stage, wh, p.out2, p.ldo2, row0, col0, p.M, p.N, p.stream_out);
  } else if constexpr (EPI == OFK_EPI_GATE_RESID_F32 || EPI == OFK_EPI_BIAS_RESID_F32) {
    // out = branch * tanh(gate) + residual (fp32 residual stream); branch kept in bf16 for the gate grad.
    uint32_t* r = aux_row;   // this lane's 32 residual values (prefetched one round ahead)
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = bf16_round(v[i]);
    if (p.out2 != nullptr) {
      uint32_t wb[16];
      pack32_bf16(v, wb);
      warp_store_tile<2, 0>(stage, wb, p.out2, p.ldo2, row0, col0, p.M, p.N, p.stream_out);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(fmaf(v[i], gate_t, __uint_as_float(r[i])));
    warp_store_tile<4, 0>(stage, r, p.out, p.ldo, row0, col0, p.M, p.N, p.stream_out);
  } else if constexpr (EPI == OFK_EPI_DGELU_BF16) {
    // out = bf16( bf16(acc) * gelu'(z) ), z = saved bf16 pre-activation
    uint32_t w[16];
    const uint32_t* z = aux_row;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      v[2 * i] = bf16_round(v[2 * i]) * gelu_exact_grad(bf16_lo(z[i]));
      v[2 * i + 1] = bf16_round(v[2 * i + 1]) * gelu_exact_grad(bf16_hi(z[i]));
    }
    pack32_bf16(v, w);
    warp_store_tile<2, 0>(stage, w, p.out, p.ldo, row0, col0, p.M, p.N, p.stream_out, p.out_rpg, p.out_gs, p.out_go);
  } else if constexpr (EPI == OFK_EPI_SWIGLU_DUAL) {
    // columns [col0, col0+16) are gate rows, [col0+16, col0+32) the matching up rows (OFK_SWIGLU_GROUP packing):
    // h = bf16(bf16(silu(g)) * u) for the 16 columns [col0/2, col0/2+16) of out, as HF LlamaMLP under autocast
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = bf16_round(v[i]);
    if (p.out2 != nullptr) {
      uint32_t wgu[16];
      pack32_bf16(v, wgu);
      warp_store_tile<2, 0>(stage, wgu, p.out2, p.ldo2, row0, col0, p.M, p.N, p.stream_out);
    }
    uint32_t wh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      wh[i] = pack_bf16x2(bf16_round(silu(v[2 * i])) * v[16 + 2 * i], bf16_round(silu(v[2 * i + 1])) * v[17 + 2 * i]);
    warp_store_tile16_bf16(stage, wh, p.out, p.ldo, row0, col0 / 2, p.M, p.N / 2, p.stream_out);
  }
}

// ----------------------------------------------------------------------------------------------
template <int BN, int A_MN, int B_MN, int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
            const GemmParams p) {
  using L = SmemLayout<BN>;
  constexpr int STAGES = L::STAGES;
  constexpr uint32_t TMEM_COLS = 2 * BN;  // two accumulator stages (256 or 512 columns)

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * L::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int m_tiles = (p.M + BM - 1) / BM;
  const int n_tiles = (p.N + BN - 1) / BN;
  const int num_work = m_tiles * n_tiles * p.splits;
  const int total_kb = (p.K + BK - 1) / BK;

  if (warp == WARP_TMA && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == WARP_MMA && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], NUM_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == WARP_TMEM) {
    tmem_alloc(tmem_ptr, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == WARP_TMA) {
    // ===================== TMA producer (one thread) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
        int mt, nt, ks;
        work_to_tile(w, m_tiles, n_tiles, mt, nt, ks);
        const int m0 = mt * BM, n0 = nt * BN;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(total_kb, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * L::STAGE_BYTES;
          uint8_t* sb = sa + L::A_BYTES;
          mbar_arrive_expect_tx(&full_bar[stage], L::STAGE_BYTES);
          const int k0 = kb * BK;
          if constexpr (A_MN == 0) {
            tma_load_2d(sa, &tma_a, &full_bar[stage], k0, m0);             // box {64 k, 128 rows}
          } else {
#pragma unroll
            for (int i = 0; i < BM / 64; ++i)                               // boxes {64 mn, 64 k}
              tma_load_2d(sa + i * (BK * 128), &tma_a, &full_bar[stage], m0 + 64 * i, (int)map_rows(k0, p.ak_rpg, p.ak_gs, p.ak_go));
          }
          if constexpr (B_MN == 0) {
            tma_load_2d(sb, &tma_b, &full_bar[stage], k0, n0);             // box {64 k, BN rows}
          } else {
#pragma unroll
            for (int i = 0; i < BN / 64; ++i)
              tma_load_2d(sb + i * (BK * 128), &tma_b, &full_bar[stage], n0 + 64 * i, k0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == WARP_MMA) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, A_MN, B_MN);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
        const int ks = w / (m_tiles * n_tiles);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(total_kb, kb0 + p.kb_per_split);
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * L::STAGE_BYTES);
          const uint32_t sb = sa + L::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // K-major : 8-row groups 1024 B apart (SBO); advance 32 B per UMMA_K inside the swizzle atom.
            // MN-major: 64-wide MN chunks BK*128 B apart (LBO), 8-k groups 1024 B apart (SBO);
            //           advance 2 k-groups = 2048 B per UMMA_K.
            const uint64_t adesc = A_MN ? make_smem_desc_sw128(sa + k * 2048, BK * 128, 1024)
                                        : make_smem_desc_sw128(sa + k * 32, 0, 1024);
            const uint64_t bdesc = B_MN ? make_smem_desc_sw128(sb + k * 2048, BK * 128, 1024)
                                        : make_smem_desc_sw128(sb + k * 32, 0, 1024);
            umma_bf16(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[as]);       // accumulator ready for the epilogue
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp < NUM_EPI_WARPS) {
    // ===================== epilogue (8 warps; TMEM -> regs -> fused op -> global) =====================
    const int q = warp & 3;                    // TMEM lane quarter == warp % 4
    const int half = warp >> 2;                // which half of the tile's columns this warp drains
    float gate_t = 1.0f;
    if constexpr (EPI == OFK_EPI_GATE_RESID_F32) {
      if (p.gate != nullptr) gate_t = tanhf(__ldg(p.gate));
    }
    int as = 0; uint32_t aphase = 0;
    for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
      int mt, nt, ks_unused;
      work_to_tile(w, m_tiles, n_tiles, mt, nt, ks_unused);
      const int n0 = nt * BN;
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * BN + half * (BN / 2);
      const uint32_t stage_addr = smem_u32(smem + STAGES * L::STAGE_BYTES + L::BAR_BYTES) + warp * STAGE_BYTES_PER_WARP;
      const int row0 = mt * BM + q * 32;
      constexpr int AUXB = AuxBytes<EPI>::value;
      uint4 pre[AUXB ? AUXB * 2 : 1];
      const int colbase = n0 + half * (BN / 2);
      if constexpr (AUXB != 0) {
        if (row0 < p.M && colbase < p.N) aux_prefetch<AUXB>(pre, p.aux, p.ldaux, row0, colbase, p.M, p.N);
      }
#pragma unroll 1
      for (int c = 0; c < BN / 64; ++c) {      // 32 columns per round: two TMEM loads in flight per wait
        uint32_t acc[32];
        tmem_ld16(taddr + c * 32, *reinterpret_cast<uint32_t(*)[16]>(&acc[0]));
        tmem_ld16(taddr + c * 32 + 16, *reinterpret_cast<uint32_t(*)[16]>(&acc[16]));
        const int col = colbase + c * 32;
        const bool live = row0 < p.M && col < p.N;                                   // warp-uniform
        uint32_t aux_row[AUXB ? AUXB * 8 : 1];
        if constexpr (AUXB != 0) {
          if (live) aux_commit<AUXB>(stage_addr, pre, aux_row);
          if (c + 1 < BN / 64 && row0 < p.M && col + 32 < p.N)                  // next round's operand: in flight
            aux_prefetch<AUXB>(pre, p.aux, p.ldaux, row0, col + 32, p.M, p.N);       // during this round's math+stores
        }
        tmem_ld_wait();
        if (live) epilogue32<EPI>(p, gate_t, stage_addr, row0, col, acc, aux_row);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_TMEM) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------------
// 2-CTA variant: a cluster of two CTAs (one SM pair) owns a 256 x 256 output tile.  Each CTA stages its own
// 128 rows of A and 128 rows of B (half the B traffic per SM of the 1-CTA kernel, so the shared-memory port
// no longer caps the tensor pipe); the leader CTA's MMA thread issues tcgen05.mma.cta_group::2 (M = 256) and
// each CTA's TMEM receives its own 128 accumulator rows, drained by its own epilogue warps.
struct Smem2 {
  static constexpr int A_BYTES = BM * BK * 2;        // 16 KiB : this CTA's 128 rows of A
  static constexpr int B_BYTES = 128 * BK * 2;       // 16 KiB : this CTA's 128 rows of B
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
#ifndef OFK_EPI_WARPS2
#define OFK_EPI_WARPS2 12
#endif
#ifndef OFK_EPI_WARPS2_RESID
#define OFK_EPI_WARPS2_RESID 8
#endif
  static constexpr int BAR_BYTES = 256;
};
// Epilogue warps of the 2-CTA kernel.  A lane quarter's 256 accumulator columns are 8 rounds of 32; with EW warps the
// EW / 4 warps of a quarter take the rounds round-robin (8 warps: 4 rounds each; 12: 3 / 3 / 2; 16: 2 each).  More warps
// per scheduler hide the tcgen05.ld -> staging -> math -> staging -> global chain of a round behind each other; the
// register budget per thread shrinks accordingly (8 warps: 168, 12: 128), which the fp32-residual epilogues feel first
// (OFK_EPI_WARPS2_RESID picks their count separately).  Same-box A/B over the 751 GEMM launches of an OF-3B step
// (tools/bench_gemm_step.py, profiles/r02_gemm_epilogue_warps.md): 8 warps everywhere 83.7 ms; 12 everywhere 83.9-85.6 ms
// (GELU / dGELU / QuickGELU epilogues 3-8 % faster, fp32-residual ones 6-17 % slower); 16 everywhere 86.3 ms; 12 for the
// math epilogues + 8 for the residual ones 83.3 ms -- the default.  The TMA ring is 6 stages with 8 epilogue warps and 5 with more
// (the per-warp staging tiles take the 32 KiB; round 1 measured 5 and 6 stages equal at K = 8192: 1621 vs ~1620 TF/s).
template <int EPI>
struct Epi2Cfg {
  static constexpr bool RESID = EPI == OFK_EPI_GATE_RESID_F32 || EPI == OFK_EPI_BIAS_RESID_F32;
  static constexpr int EW = RESID ? OFK_EPI_WARPS2_RESID : OFK_EPI_WARPS2;
  static constexpr int THREADS = (EW + 4) * 32;
  static constexpr int WARP_TMA = EW, WARP_MMA = EW + 1, WARP_TMEM = EW + 2;
  static constexpr int STAGES = EW <= 8 ? 6 : 5;
  static constexpr int TOTAL = STAGES * Smem2::STAGE_BYTES + Smem2::BAR_BYTES + EW * 32 * 128 + 1024;
};

template <int A_MN, int B_MN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Epi2Cfg<EPI>::THREADS, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
             const GemmParams p) {
  using L = Smem2;
  using E = Epi2Cfg<EPI>;
  constexpr int STAGES = E::STAGES;
  constexpr int EPI_WARPS2 = E::EW;
  constexpr int BN2 = 256;
  constexpr uint32_t TMEM_COLS = 2 * BN2;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * L::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;

  const int m_tiles = (p.M + 255) / 256;
  const int n_tiles = (p.N + BN2 - 1) / BN2;
  const int total_kb = (p.K + BK - 1) / BK;
  const int num_work = p.tail_s > 0 ? p.tail_first + (m_tiles * n_tiles - p.tail_first) * p.tail_s
                                    : m_tiles * n_tiles * p.splits;
  const int first_work = (int)cluster_id_x();
  const int work_stride = (int)num_clusters_x();

  if (warp == E::WARP_TMA && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == E::WARP_MMA && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * EPI_WARPS2); }  // both CTAs' warps
    fence_barrier_init();
  }
  if (warp == E::WARP_TMEM) {
    tmem_alloc_2cta(tmem_ptr, TMEM_COLS);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // peer barriers are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == E::WARP_TMA) {
    // ===================== TMA producer (one thread per CTA) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int w = first_work; w < num_work; w += work_stride) {
        const Work2 wk = decode_work2(p, w, m_tiles, n_tiles, total_kb);
        const int m0 = wk.mt * 256 + (int)cta_rank * 128;
        const int n0 = wk.nt * BN2 + (int)cta_rank * 128;
        const int kb0 = wk.kb0, kb1 = wk.kb1;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * L::STAGE_BYTES;
          uint8_t* sb = sa + L::A_BYTES;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * L::STAGE_BYTES);  // both CTAs' bytes land here
          const int k0 = kb * BK;
          if constexpr (A_MN == 0) {
            tma_load_2d_2cta(sa, &tma_a, &full_bar[stage], k0, m0);
          } else {
#pragma unroll
            for (int i = 0; i < 2; ++i)
              tma_load_2d_2cta(sa + i * (BK * 128), &tma_a, &full_bar[stage], m0 + 64 * i, (int)map_rows(k0, p.ak_rpg, p.ak_gs, p.ak_go));
          }
          if constexpr (B_MN == 0) {
            tma_load_2d_2cta(sb, &tma_b, &full_bar[stage], k0, n0);
          } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) tma_load_2d_2cta(sb + i * (BK * 128), &tma_b, &full_bar[stage], n0 + 64 * i, k0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == E::WARP_MMA) {
    // ===================== MMA issuer (one thread of the leader CTA) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(256, BN2, A_MN, B_MN);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      for (int w = first_work; w < num_work; w += work_stride) {
        const Work2 wk = decode_work2(p, w, m_tiles, n_tiles, total_kb);
        const int kb0 = wk.kb0, kb1 = wk.kb1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN2;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * L::STAGE_BYTES);
          const uint32_t sb = sa + L::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = A_MN ? make_smem_desc_sw128(sa + k * 2048, BK * 128, 1024)
                                        : make_smem_desc_sw128(sa + k * 32, 0, 1024);
            const uint64_t bdesc = B_MN ? make_smem_desc_sw128(sb + k * 2048, BK * 128, 1024)
                                        : make_smem_desc_sw128(sb + k * 32, 0, 1024);
            umma_bf16_2cta(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit_2cta(&empty_bar[stage]);   // frees this stage in BOTH CTAs
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2cta(&tmem_full[as]);        // accumulator ready in BOTH CTAs
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp < EPI_WARPS2) {
    // ===================== epilogue (EPI_WARPS2 warps per CTA; this CTA's 128 rows) =====================
    const int q = warp & 3;                    // TMEM lane quarter == warp % 4
    const int t3 = warp >> 2;                  // which of the quarter's warps: takes rounds t3, t3 + W, t3 + 2W, ...
    constexpr int WPQ = EPI_WARPS2 / 4;        // warps per quarter
    float gate_t = 1.0f;
    if constexpr (EPI == OFK_EPI_GATE_RESID_F32) {
      if (p.gate != nullptr) gate_t = tanhf(__ldg(p.gate));
    }
    int as = 0; uint32_t aphase = 0;
    for (int w = first_work; w < num_work; w += work_stride) {
      const Work2 wk = decode_work2(p, w, m_tiles, n_tiles, total_kb);
      const int mt = wk.mt, nt = wk.nt;
      const int n0 = nt * BN2;
      // tail-split partials / flags are indexed per (CTA, lane quarter, round): one producer and one consumer warp each
      const int fslot = (int)cta_rank * 32 + q * 8;
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * BN2;
      if (wk.role == 1) {
        // ---- tail-split producer: dump this warp's rounds (32 x 32 fp32 each) in register order, then signal per round
#pragma unroll 1
        for (int r = t3; r < BN2 / 32; r += WPQ) {
          float* wsp = p.tail_ws + ((size_t)(wk.t * (p.tail_s - 1) + wk.j) * 64 + fslot + r) * 1024 + lane * 4;
          uint32_t acc[32];
          tmem_ld16(taddr + r * 32, *reinterpret_cast<uint32_t(*)[16]>(&acc[0]));
          tmem_ld16(taddr + r * 32 + 16, *reinterpret_cast<uint32_t(*)[16]>(&acc[16]));
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 8; ++i)
            st_global_cg_v4(wsp + i * 128, make_uint4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]));
          __threadfence();
          __syncwarp();
          if (lane == 0) {
            __threadfence();
            atomicAdd(p.tail_flags + wk.t * 64 + fslot + r, 1);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&tmem_empty[as], 0);
        if (++as == 2) { as = 0; aphase ^= 1; }
        continue;
      }
      const uint32_t stage_addr = smem_u32(smem + STAGES * L::STAGE_BYTES + L::BAR_BYTES) + warp * STAGE_BYTES_PER_WARP;
      const int row0 = mt * 256 + (int)cta_rank * 128 + q * 32;
      constexpr int AUXB = AuxBytes<EPI>::value;
      uint4 pre[AUXB ? AUXB * 2 : 1];
      if constexpr (AUXB != 0) {
        if (row0 < p.M && n0 + t3 * 32 < p.N) aux_prefetch<AUXB>(pre, p.aux, p.ldaux, row0, n0 + t3 * 32, p.M, p.N);
      }
#pragma unroll 1
      for (int r = t3; r < BN2 / 32; r += WPQ) {      // 32 columns per round: two TMEM loads in flight per wait
        uint32_t acc[32];
        tmem_ld16(taddr + r * 32, *reinterpret_cast<uint32_t(*)[16]>(&acc[0]));
        tmem_ld16(taddr + r * 32 + 16, *reinterpret_cast<uint32_t(*)[16]>(&acc[16]));
        const int col = n0 + r * 32;
        const bool live = row0 < p.M && col < p.N;                                   // warp-uniform
        uint32_t aux_row[AUXB ? AUXB * 8 : 1];
        if constexpr (AUXB != 0) {
          if (live) aux_commit<AUXB>(stage_addr, pre, aux_row);
          if (r + WPQ < BN2 / 32 && row0 < p.M && col + WPQ * 32 < p.N)              // next round's operand: in flight
            aux_prefetch<AUXB>(pre, p.aux, p.ldaux, row0, col + WPQ * 32, p.M, p.N); // during this round's math+stores
        }
        tmem_ld_wait();
        if (wk.role == 2) {
          // ---- tail-split owner: wait until the other slices' partials for this (quarter, round) have landed
          int* flag = p.tail_flags + wk.t * 64 + fslot + r;
          if (lane == 0) {
            while (ld_acquire_gpu(flag) < p.tail_s - 1) __nanosleep(64);
            *flag = 0;                                   // single consumer: ready for the next launch
          }
          __syncwarp();
          __threadfence();
          const float* wsp = p.tail_ws + ((size_t)(wk.t * (p.tail_s - 1)) * 64 + fslot + r) * 1024 + lane * 4;
          for (int j = 0; j < p.tail_s - 1; ++j) {
            const float* pj = wsp + (size_t)j * 64 * 1024;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint4 u = ld_global_cg_v4(pj + i * 128);
              acc[4 * i] = __float_as_uint(__uint_as_float(acc[4 * i]) + __uint_as_float(u.x));
              acc[4 * i + 1] = __float_as_uint(__uint_as_float(acc[4 * i + 1]) + __uint_as_float(u.y));
              acc[4 * i + 2] = __float_as_uint(__uint_as_float(acc[4 * i + 2]) + __uint_as_float(u.z));
              acc[4 * i + 3] = __float_as_uint(__uint_as_float(acc[4 * i + 3]) + __uint_as_float(u.w));
            }
          }
        }
        if (live) epilogue32<EPI>(p, gate_t, stage_addr, row0, col, acc, aux_row);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tmem_empty[as], 0);   // the leader's MMA thread waits for all 2 x EPI_WARPS2 warps
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // neither CTA may free TMEM / exit while its peer can still touch it
  if (warp == E::WARP_TMEM) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------------
// Host side: tensor-map cache + dispatch.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  });
  return fn;
}

struct MapKey {
  const void* ptr; long long ld; int rows, cols, box_inner, box_outer;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && ld == o.ld && rows == o.rows && cols == o.cols && box_inner == o.box_inner &&
           box_outer == o.box_outer;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ (size_t)k.ld; h = h * 1000003u ^ (size_t)k.rows; h = h * 1000003u ^ (size_t)k.cols;
    h = h * 1000003u ^ (size_t)(k.box_inner * 1024 + k.box_outer);
    return h;
  }
};

// 2-D bf16 row-major tensor [rows, cols] (cols contiguous, row stride ld elements), 128B swizzle.
static int get_tensor_map(const void* ptr, long long ld, int rows, int cols, int box_inner, int box_outer,
                          CUtensorMap* out) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{ptr, ld, rows, cols, box_inner, box_outer};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return ofk_set_error(OFK_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not found");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * 2) & 15))
    return ofk_set_error(OFK_ERR_ALIGN, "GEMM operand must be 16-byte aligned with a 16-byte-multiple row stride");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[160];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%lld box=%dx%d", (int)r, rows,
             cols, ld, box_inner, box_outer);
    return ofk_set_error(OFK_ERR_DRIVER, buf);
  }
  {
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > 4096) cache.clear();
    cache.emplace(key, m);
  }
  *out = m;
  return 0;
}

static int g_num_sms = 0;
static int g_reserved_sms = 0;   // SMs the persistent grids leave free (ofk_gemm_reserve_sms): room for NCCL's CTAs

template <int BN, int A_MN, int B_MN, int EPI>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, cudaStream_t stream) {
  using L = SmemLayout<BN>;
  auto kern = gemm_kernel<BN, A_MN, B_MN, EPI>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
    if (e != cudaSuccess) return ofk_set_error(OFK_ERR_CUDA, cudaGetErrorString(e));
    attr_done = true;
  }
  const int m_tiles = (p.M + BM - 1) / BM, n_tiles = (p.N + BN - 1) / BN;
  const int work = m_tiles * n_tiles * p.splits;
  const int avail = g_num_sms - g_reserved_sms;
  const int grid = work < avail ? work : avail;
  kern<<<grid, NUM_THREADS, L::TOTAL, stream>>>(ta, tb, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return ofk_set_error(OFK_ERR_CUDA, cudaGetErrorString(e));
  ofk_count_launch();
  return 0;
}

template <int A_MN, int B_MN, int EPI>
static int launch2(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, cudaStream_t stream) {
  auto kern = gemm2_kernel<A_MN, B_MN, EPI>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Epi2Cfg<EPI>::TOTAL);
    if (e != cudaSuccess) return ofk_set_error(OFK_ERR_CUDA, cudaGetErrorString(e));
    attr_done = true;
  }
  const int tiles2 = ((p.M + 255) / 256) * ((p.N + 255) / 256);
  const int work = p.tail_s > 0 ? p.tail_first + (tiles2 - p.tail_first) * p.tail_s : tiles2 * p.splits;
  int clusters = (g_num_sms - g_reserved_sms) / 2;
  if (work < clusters) clusters = work;
  kern<<<2 * clusters, Epi2Cfg<EPI>::THREADS, Epi2Cfg<EPI>::TOTAL, stream>>>(ta, tb, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return ofk_set_error(OFK_ERR_CUDA, cudaGetErrorString(e));
  ofk_count_launch();
  return 0;
}

template <int EPI>
static int dispatch_major2(int a_mn, int b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
                           cudaStream_t s) {
  if (a_mn == 0 && b_mn == 0) return launch2<0, 0, EPI>(ta, tb, p, s);
  if (a_mn == 0 && b_mn == 1) return launch2<0, 1, EPI>(ta, tb, p, s);
  if (a_mn == 1 && b_mn == 1) return launch2<1, 1, EPI>(ta, tb, p, s);
  return launch2<1, 0, EPI>(ta, tb, p, s);
}

static int dispatch_epi2(int epi, int a_mn, int b_mn, const CUtensorMap& ta, const CUtensorMap& tb,
                         const GemmParams& p, cudaStream_t s) {
  switch (epi) {
    case OFK_EPI_STORE_BF16: return dispatch_major2<OFK_EPI_STORE_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_STORE_F32: return dispatch_major2<OFK_EPI_STORE_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_ATOMIC_F32: return dispatch_major2<OFK_EPI_ATOMIC_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_BF16: return dispatch_major2<OFK_EPI_BIAS_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_QGELU_BF16: return dispatch_major2<OFK_EPI_BIAS_QGELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_GELU_DUAL: return dispatch_major2<OFK_EPI_GELU_DUAL>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_GATE_RESID_F32: return dispatch_major2<OFK_EPI_GATE_RESID_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_DGELU_BF16: return dispatch_major2<OFK_EPI_DGELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_RESID_F32: return dispatch_major2<OFK_EPI_BIAS_RESID_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_GELU_BF16: return dispatch_major2<OFK_EPI_BIAS_GELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_SWIGLU_DUAL: return launch2<0, 0, OFK_EPI_SWIGLU_DUAL>(ta, tb, p, s);   // K-major only (gemm_impl)
  }
  return ofk_set_error(OFK_ERR_ARG, "unknown GEMM epilogue");
}

template <int BN, int EPI>
static int dispatch_major(int a_mn, int b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
                          cudaStream_t s) {
  if (a_mn == 0 && b_mn == 0) return launch<BN, 0, 0, EPI>(ta, tb, p, s);
  if (a_mn == 0 && b_mn == 1) return launch<BN, 0, 1, EPI>(ta, tb, p, s);
  if (a_mn == 1 && b_mn == 1) return launch<BN, 1, 1, EPI>(ta, tb, p, s);
  return launch<BN, 1, 0, EPI>(ta, tb, p, s);
}

template <int BN>
static int dispatch_epi(int epi, int a_mn, int b_mn, const CUtensorMap& ta, const CUtensorMap& tb,
                        const GemmParams& p, cudaStream_t s) {
  switch (epi) {
    case OFK_EPI_STORE_BF16: return dispatch_major<BN, OFK_EPI_STORE_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_STORE_F32: return dispatch_major<BN, OFK_EPI_STORE_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_ATOMIC_F32: return dispatch_major<BN, OFK_EPI_ATOMIC_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_BF16: return dispatch_major<BN, OFK_EPI_BIAS_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_QGELU_BF16: return dispatch_major<BN, OFK_EPI_BIAS_QGELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_GELU_DUAL: return dispatch_major<BN, OFK_EPI_GELU_DUAL>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_GATE_RESID_F32: return dispatch_major<BN, OFK_EPI_GATE_RESID_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_DGELU_BF16: return dispatch_major<BN, OFK_EPI_DGELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_RESID_F32: return dispatch_major<BN, OFK_EPI_BIAS_RESID_F32>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_BIAS_GELU_BF16: return dispatch_major<BN, OFK_EPI_BIAS_GELU_BF16>(a_mn, b_mn, ta, tb, p, s);
    case OFK_EPI_SWIGLU_DUAL: return launch<BN, 0, 0, OFK_EPI_SWIGLU_DUAL>(ta, tb, p, s);
  }
  return ofk_set_error(OFK_ERR_ARG, "unknown GEMM epilogue");
}

}  // namespace ofk

int ofk_tensor_map_bf16(const void* ptr, long long ld, int rows, int cols, int box_inner, int box_outer,
                        struct CUtensorMap_st* out) {
  return ofk::get_tensor_map(ptr, ld, rows, cols, box_inner, box_outer, out);
}

// Tail-split workspace: 4 KiB of per-warp flags (zero before first use; self-resetting) + one 256 x 256 fp32
// partial per producer slice.  rem <= P / 2 = 37 tiles and rem * (s - 1) < P = 74 partials on a 148-SM part.
constexpr int OFK_GEMM_WS_TILES = 74;
constexpr long long OFK_GEMM_WS_FLAG_BYTES = 16384;   // 64 flags (2 CTAs x 4 lane quarters x 8 rounds) per tail tile, <= 37 tiles
constexpr long long OFK_GEMM_WS_BYTES = OFK_GEMM_WS_FLAG_BYTES + (long long)OFK_GEMM_WS_TILES * 256 * 256 * 4;
constexpr int TAIL_MIN_KB = 48;   // below ~3k of K half a tile-time is not worth the partial round trip
static bool tail_split_enabled() {
  static int mode = -1;
  if (mode < 0) { const char* e = getenv("OFK_GEMM_TAIL_SPLIT"); mode = e ? (atoi(e) != 0) : 1; }
  return mode == 1;
}

static int gemm_impl(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                     long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                     void* out2, long long ldo2, const void* aux, long long ldaux, const float* bias,
                     const float* gate, void* stream_, int out_rpg, int out_gs, int out_go, int ak_rpg, int ak_gs,
                     int ak_go, void* workspace = nullptr, long long workspace_bytes = 0) {
  using namespace ofk;
  if (out_rpg > 0 && (epi != OFK_EPI_STORE_BF16 && epi != OFK_EPI_BIAS_BF16 && epi != OFK_EPI_STORE_F32))
    return ofk_set_error(OFK_ERR_ARG, "grouped output rows are supported by the STORE_BF16 / BIAS_BF16 / STORE_F32 epilogues");
  if (ak_rpg > 0 && (!a_mn_major || ak_rpg % 64 != 0 || K % ak_rpg != 0))
    return ofk_set_error(OFK_ERR_ARG, "grouped reduction rows need an MN-major A with rows_per_group % 64 == 0 dividing K");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (M <= 0 || N <= 0 || K <= 0) return ofk_set_error(OFK_ERR_ARG, "GEMM dims must be positive");
  if (N % 16 != 0) return ofk_set_error(OFK_ERR_ARG, "GEMM N must be a multiple of 16");
  if (!A || !B || !out) return ofk_set_error(OFK_ERR_ARG, "GEMM null operand");
  if (splits < 1) splits = 1;
  if (splits > 1 && epi != OFK_EPI_ATOMIC_F32) return ofk_set_error(OFK_ERR_ARG, "split-K needs the atomic epilogue");
  if ((epi == OFK_EPI_BIAS_BF16 || epi == OFK_EPI_BIAS_QGELU_BF16 || epi == OFK_EPI_BIAS_RESID_F32 ||
       epi == OFK_EPI_BIAS_GELU_BF16) && !bias)
    return ofk_set_error(OFK_ERR_ARG, "bias epilogue without bias");
  if ((epi == OFK_EPI_GATE_RESID_F32 || epi == OFK_EPI_BIAS_RESID_F32 || epi == OFK_EPI_DGELU_BF16) && !aux)
    return ofk_set_error(OFK_ERR_ARG, "epilogue needs aux operand");
  if (epi == OFK_EPI_GELU_DUAL && !out2) return ofk_set_error(OFK_ERR_ARG, "GELU_DUAL needs out2");
  if (epi == OFK_EPI_SWIGLU_DUAL && (a_mn_major || b_mn_major || N % (2 * OFK_SWIGLU_GROUP) != 0 || splits > 1 || out_rpg > 0))
    return ofk_set_error(OFK_ERR_ARG, "SWIGLU_DUAL needs K-major A and B, N % 32 == 0 and no split-K");
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) return ofk_set_error(OFK_ERR_CUDA, "no CUDA device");
  }
  // block_n: 0 = auto, 128 / 256 = 1-CTA tile width, 512 = force the 2-CTA (256 x 256 per SM pair) kernel
  const bool two_cta = block_n == 512 || (block_n == 0 && M >= 512 && N >= 256);
  const int BN = (block_n == 128 || block_n == 256) ? block_n : ((N % 256 == 0 || N > 1024) ? 256 : 128);
  const int total_kb = (K + BK - 1) / BK;
  if (splits > total_kb) splits = total_kb;
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.kb_per_split = (total_kb + splits - 1) / splits;
  p.splits = (total_kb + p.kb_per_split - 1) / p.kb_per_split;
  p.out = out; p.ldo = ldo; p.out2 = out2; p.ldo2 = ldo2; p.aux = aux; p.ldaux = ldaux; p.bias = bias; p.gate = gate;
  p.out_rpg = out_rpg; p.out_gs = out_gs; p.out_go = out_go; p.ak_rpg = ak_rpg; p.ak_gs = ak_gs; p.ak_go = ak_go;
  p.tail_first = 0; p.tail_s = 0; p.tail_kps = 0; p.tail_ws = nullptr; p.tail_flags = nullptr;
  if (two_cta && p.splits == 1 && epi != OFK_EPI_ATOMIC_F32 && workspace != nullptr &&
      workspace_bytes >= OFK_GEMM_WS_BYTES && tail_split_enabled() && total_kb >= TAIL_MIN_KB) {
    // The persistent grid walks `tiles` 256 x 256 tiles on P SM pairs; when the last round is at most half full,
    // cut its tiles into k-slices so that round costs 1/s of a tile-time (plus one fp32 partial round trip
    // through L2) instead of a whole one: e.g. the N = 2048 GEMMs of MPT-1B are 256 tiles on 74 pairs = 3.46 rounds.
    const int P = (g_num_sms - g_reserved_sms) / 2;
    const int tiles = ((M + 255) / 256) * ((N + 255) / 256);
    const int rem = tiles % P;
    if (rem > 0 && rem <= OFK_GEMM_WS_TILES / 2) {
      int s_ = P / rem;
      if (s_ > 4) s_ = 4;
      if (s_ > total_kb / 16) s_ = total_kb / 16;
      if (s_ >= 2 && rem * (s_ - 1) <= OFK_GEMM_WS_TILES) {
        p.tail_first = tiles - rem;
        p.tail_s = s_;
        p.tail_kps = (total_kb + s_ - 1) / s_;
        p.tail_flags = reinterpret_cast<int*>(workspace);
        p.tail_ws = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + OFK_GEMM_WS_FLAG_BYTES);
      }
    }
  }
  const int a_rows = ak_rpg > 0 ? (K / ak_rpg) * ak_gs : K;   // physical row count of an MN-major A
  {
    static int stream_mode = -1;   // OFK_GEMM_STREAM_OUT=0/1 overrides; default: stream when the outputs exceed ~32 MB
    if (stream_mode < 0) { const char* e = getenv("OFK_GEMM_STREAM_OUT"); stream_mode = e ? atoi(e) + 2 : 0; }
    if (stream_mode >= 2) p.stream_out = stream_mode - 2;
    else p.stream_out = ((long long)M * N >= (16LL << 20)) ? 1 : 0;
  }

  CUtensorMap ta, tb;
  int rc;
  if (two_cta) {
    rc = a_mn_major ? get_tensor_map(A, lda, a_rows, M, 64, BK, &ta) : get_tensor_map(A, lda, M, K, BK, 128, &ta);
    if (rc) return rc;
    rc = b_mn_major ? get_tensor_map(B, ldb, K, N, 64, BK, &tb) : get_tensor_map(B, ldb, N, K, BK, 128, &tb);
    if (rc) return rc;
    return dispatch_epi2(epi, a_mn_major, b_mn_major, ta, tb, p, stream);
  }
  // K-major: tensor [rows, K], box {64 (k), tile rows}. MN-major: tensor [K, rows], box {64 (rows), 64 (k)}.
  rc = a_mn_major ? get_tensor_map(A, lda, a_rows, M, 64, BK, &ta) : get_tensor_map(A, lda, M, K, BK, BM, &ta);
  if (rc) return rc;
  rc = b_mn_major ? get_tensor_map(B, ldb, K, N, 64, BK, &tb) : get_tensor_map(B, ldb, N, K, BK, BN, &tb);
  if (rc) return rc;
  if (BN == 256) return dispatch_epi<256>(epi, a_mn_major, b_mn_major, ta, tb, p, stream);
  return dispatch_epi<128>(epi, a_mn_major, b_mn_major, ta, tb, p, stream);
}

extern "C" int ofk_gemm_bf16(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                             long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                             void* out2, long long ldo2, const void* aux, long long ldaux, const float* bias,
                             const float* gate, void* stream_) {
  return gemm_impl(epi, a_mn_major, b_mn_major, A, lda, B, ldb, M, N, K, splits, block_n, out, ldo, out2, ldo2, aux, ldaux,
                   bias, gate, stream_, 0, 0, 0, 0, 0, 0);
}

extern "C" long long ofk_gemm_workspace_bytes(void) { return OFK_GEMM_WS_BYTES; }

extern "C" int ofk_gemm_reserve_sms(int n) {
  const int prev = ofk::g_reserved_sms;
  if (n < 0) n = 0;
  if (n > 64) n = 64;
  ofk::g_reserved_sms = n & ~1;   // whole SM pairs
  return prev;
}

extern "C" int ofk_gemm_bf16_ws(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                                long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                                void* out2, long long ldo2, const void* aux, long long ldaux, const float* bias,
                                const float* gate, void* workspace, long long workspace_bytes, void* stream_) {
  return gemm_impl(epi, a_mn_major, b_mn_major, A, lda, B, ldb, M, N, K, splits, block_n, out, ldo, out2, ldo2, aux, ldaux,
                   bias, gate, stream_, 0, 0, 0, 0, 0, 0, workspace, workspace_bytes);
}

extern "C" int ofk_gemm_bf16_grouped(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                                     long long ldb, int M, int N, int K, int splits, int block_n, void* out,
                                     long long ldo, const float* bias, int out_rows_per_group, int out_group_stride,
                                     int out_group_offset, int a_k_rows_per_group, int a_k_group_stride,
                                     int a_k_group_offset, void* stream_) {
  return gemm_impl(epi, a_mn_major, b_mn_major, A, lda, B, ldb, M, N, K, splits, block_n, out, ldo, nullptr, 0, nullptr, 0,
                   bias, nullptr, stream_, out_rows_per_group, out_group_stride, out_group_offset, a_k_rows_per_group,
                   a_k_group_stride, a_k_group_offset);
}
