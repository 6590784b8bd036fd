// Fused self-attention for BERT geometry (S = 128 keys per sequence, head_dim = 64) on tcgen05.
// Every other sequence length and head size goes to the tiled kernels (attention_tiled_sm100.cu).
//
// One CTA per (batch, head).  With S = 128 a whole score matrix is exactly one 128x128 UMMA tile,
// so no online-softmax tiling is needed:
//
//   forward : S = Q K^T (UMMA 128x128x64)  -> TMEM -> per-row softmax (+mask, +dropout) in
//             registers -> P (bf16) into swizzled smem -> O = P V (UMMA 128x64x128) -> ctx
//   backward: S = Q K^T, dP = dO V^T -> registers: P = exp2(s - lse), dS = P (dP*keep - delta)
//             -> smem (one copy serves as K-major AND MN-major operand) ->
//             dV = P^T dO, dK = dS^T Q, dQ = dS K  (three UMMAs, accumulators side by side in TMEM)
//
// Q/K/V/dO tiles come straight out of the fused [tokens, 3H] QKV activation via 2D TMA boxes
// (no head split/merge copies), outputs are written head-merged.
//
// Reference parity: BertSelfAttention.forward, scaelum/model/bert_layers.py:249-275 (scores /
// sqrt(d) + mask, softmax, dropout on probabilities, P V, head merge) and its autograd backward.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdlib>

#include "api.h"
#include "launch_util.h"
#include "sm100_ptx.cuh"

namespace sky {

int make_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t outer,
                      uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer);

namespace {

constexpr int kS = 128;   // sequence length handled by this kernel
constexpr int kD = 64;    // head dim
constexpr int kTile = kS * kD * 2;  // 16 KB: one [128 x 64] bf16 tile
constexpr float kLog2e = 1.4426950408889634f;

// byte offset of element (row, col) inside a [128 x 64]-bf16 SWIZZLE_128B tile (16B granularity)
__device__ __forceinline__ uint32_t sw128_offset(int row, int col) {
  const uint32_t chunk = static_cast<uint32_t>(col >> 3) ^ static_cast<uint32_t>(row & 7);
  return static_cast<uint32_t>(row) * 128u + (chunk << 4) + static_cast<uint32_t>(col & 7) * 2u;
}

struct AttnDev {
  const float* mask;  // [B,S] additive or null
  __nv_bfloat16* ctx;
  float* lse;  // [B*heads, S] log2-domain log-sum-exp
  const __nv_bfloat16* ctx_in;
  __nv_bfloat16* dqkv;
  int heads;
  int H;  // heads * 64
  float scale;
  float dropout_p;
  const uint64_t* rng_state;
  uint32_t rng_stream;
};

// ----------------------------------------------------------------------------------------------
// forward
// ----------------------------------------------------------------------------------------------
constexpr int kFwdSmem = 3 * kTile + 2 * kTile /*P*/ + 1024 /*align*/ + 512 /*mask*/ + 64;

__global__ void __launch_bounds__(128, 2)
attention_fwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnDev p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + kTile;
  uint8_t* sV = smem + 2 * kTile;
  uint8_t* sP = smem + 3 * kTile;  // two [128 x 64] K-blocks
  float* sMask = reinterpret_cast<float*>(smem + 5 * kTile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 5 * kTile + 512);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // uniform: MMA operands stay in URs
  const int bh = blockIdx.x;
  const int b = bh / p.heads;
  const int h = bh % p.heads;

  if (tid == 0) {
    tma_prefetch_desc(&tmap_qkv);
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, 256);
    tmem_relinquish();
  }
  pdl_wait();
  pdl_launch_dependents();
  sMask[tid] = p.mask ? p.mask[b * kS + tid] * kLog2e : 0.f;
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0 && elect_one_sync()) {
    mbar_expect_tx(&bars[0], 3 * kTile);
    tma_load_2d(sQ, &tmap_qkv, &bars[0], h * kD, b * kS);
    tma_load_2d(sK, &tmap_qkv, &bars[0], p.H + h * kD, b * kS);
    tma_load_2d(sV, &tmap_qkv, &bars[0], 2 * p.H + h * kD, b * kS);
    mbar_wait(&bars[0], 0);
    tcgen05_fence_after();
    constexpr uint32_t idesc = make_idesc_bf16_f32(128, 128, false, false);
    const uint64_t da = make_smem_desc_sw128(smem_u32(sQ), 16, 1024);
    const uint64_t db = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
#pragma unroll
    for (int k = 0; k < kD / 16; ++k) umma_bf16_ss(tmem_base, da + 2 * k, db + 2 * k, idesc, k);
    umma_commit(&bars[1]);
  }
  mbar_wait(&bars[1], 0);
  tcgen05_fence_after();

  // ---- softmax over my row (query index = tid) ----
  const uint32_t trow = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
  const float sc = p.scale * kLog2e;
  float mx = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(trow + c * 32, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]) * sc + sMask[c * 32 + j]);
  }
  const bool has_dropout = p.dropout_p > 0.f;
  uint64_t seed = 0;
  uint32_t thr16 = 0;
  if (has_dropout) {
    seed = dropout_seed(p.rng_state, p.rng_stream);
    thr16 = static_cast<uint32_t>(p.dropout_p * 65536.f);
  }
  const uint64_t drop_row = (static_cast<uint64_t>(bh) * kS + tid) * kS;
  float sum = 0.f;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(trow + c * 32, v);
    tmem_ld_wait();
    float e[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      e[j] = exp2f(__uint_as_float(v[j]) * sc + sMask[c * 32 + j] - mx);
      sum += e[j];
    }
    if (has_dropout) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const uint32_t m = dropout_keep4(seed, (drop_row + c * 32 + j) >> 2, thr16);
        e[j] = (m & 1u) ? e[j] : 0.f;
        e[j + 1] = (m & 2u) ? e[j + 1] : 0.f;
        e[j + 2] = (m & 4u) ? e[j + 2] : 0.f;
        e[j + 3] = (m & 8u) ? e[j + 3] : 0.f;
      }
    }
    uint8_t* blk = sP + (c >> 1) * kTile;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      uint4 pk;
      pk.x = pack_bf16x2(e[j], e[j + 1]);
      pk.y = pack_bf16x2(e[j + 2], e[j + 3]);
      pk.z = pack_bf16x2(e[j + 4], e[j + 5]);
      pk.w = pack_bf16x2(e[j + 6], e[j + 7]);
      *reinterpret_cast<uint4*>(blk + sw128_offset(tid, (c & 1) * 32 + j)) = pk;
    }
  }
  if (p.lse != nullptr) p.lse[static_cast<long long>(bh) * kS + tid] = mx + log2f(sum);
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();

  if (warp == 0 && elect_one_sync()) {
    tcgen05_fence_after();
    constexpr uint32_t idesc = make_idesc_bf16_f32(128, 64, false, true);
#pragma unroll
    for (int j = 0; j < kS / 16; ++j) {
      const uint64_t da =
          make_smem_desc_sw128(smem_u32(sP + (j >> 2) * kTile) + (j & 3) * 32, 16, 1024);
      const uint64_t db = make_smem_desc_sw128(smem_u32(sV) + j * 2048, kTile, 1024);
      umma_bf16_ss(tmem_base + 128, da, db, idesc, j);
    }
    umma_commit(&bars[2]);
  }
  mbar_wait(&bars[2], 0);
  tcgen05_fence_after();

  const float inv = (has_dropout ? 1.f / (1.f - p.dropout_p) : 1.f) / sum;
  __nv_bfloat16* orow = p.ctx + (static_cast<long long>(b) * kS + tid) * p.H + h * kD;
#pragma unroll 1
  for (int c = 0; c < 2; ++c) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(trow + 128 + c * 32, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      uint4 pk;
      pk.x = pack_bf16x2(__uint_as_float(v[j]) * inv, __uint_as_float(v[j + 1]) * inv);
      pk.y = pack_bf16x2(__uint_as_float(v[j + 2]) * inv, __uint_as_float(v[j + 3]) * inv);
      pk.z = pack_bf16x2(__uint_as_float(v[j + 4]) * inv, __uint_as_float(v[j + 5]) * inv);
      pk.w = pack_bf16x2(__uint_as_float(v[j + 6]) * inv, __uint_as_float(v[j + 7]) * inv);
      *reinterpret_cast<uint4*>(orow + c * 32 + j) = pk;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ----------------------------------------------------------------------------------------------
// backward
// ----------------------------------------------------------------------------------------------
// 7 tiles (Q, K, V, dO, P1, dS0, dS1; P0 re-uses V once dP = dO V^T has retired) + mask + barriers:
// 115,264 B, i.e. two CTAs fit one SM (the 1024-B alignment comes from the declaration, no slack).
constexpr int kBwdSmem = 7 * kTile + 512 + 64;

__global__ void __launch_bounds__(128, 2)
attention_bwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv,
                     const __grid_constant__ CUtensorMap tmap_do, const AttnDev p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0) __trap();  // SWIZZLE_128B tiles need 1024-B alignment
  uint8_t* sQ = smem;
  uint8_t* sK = smem + kTile;
  uint8_t* sV = smem + 2 * kTile;
  uint8_t* sdO = smem + 3 * kTile;
  uint8_t* sP0 = sV;                // keys 0..63 of P: V is dead once dP has been computed
  uint8_t* sP1 = smem + 4 * kTile;  // keys 64..127 of P
  uint8_t* sdS = smem + 5 * kTile;  // 2 blocks
  float* sMask = reinterpret_cast<float*>(smem + 7 * kTile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 7 * kTile + 512);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int bh = blockIdx.x;
  const int b = bh / p.heads;
  const int h = bh % p.heads;

  if (tid == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, 256);
    tmem_relinquish();
  }
  pdl_wait();
  pdl_launch_dependents();
  sMask[tid] = p.mask ? p.mask[b * kS + tid] * kLog2e : 0.f;
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // S and dP are dead after the softmax phase: the three output accumulators re-use their columns
  constexpr uint32_t cS = 0, cdP = 128, cdV = 0, cdK = 64, cdQ = 128;

  if (warp == 0 && elect_one_sync()) {
    mbar_expect_tx(&bars[0], 4 * kTile);
    tma_load_2d(sQ, &tmap_qkv, &bars[0], h * kD, b * kS);
    tma_load_2d(sK, &tmap_qkv, &bars[0], p.H + h * kD, b * kS);
    tma_load_2d(sV, &tmap_qkv, &bars[0], 2 * p.H + h * kD, b * kS);
    tma_load_2d(sdO, &tmap_do, &bars[0], h * kD, b * kS);
    mbar_wait(&bars[0], 0);
    tcgen05_fence_after();
    constexpr uint32_t idesc = make_idesc_bf16_f32(128, 128, false, false);
    const uint64_t dq = make_smem_desc_sw128(smem_u32(sQ), 16, 1024);
    const uint64_t dk = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
    const uint64_t ddo = make_smem_desc_sw128(smem_u32(sdO), 16, 1024);
    const uint64_t dv = make_smem_desc_sw128(smem_u32(sV), 16, 1024);
#pragma unroll
    for (int k = 0; k < kD / 16; ++k)
      umma_bf16_ss(tmem_base + cS, dq + 2 * k, dk + 2 * k, idesc, k);
#pragma unroll
    for (int k = 0; k < kD / 16; ++k)
      umma_bf16_ss(tmem_base + cdP, ddo + 2 * k, dv + 2 * k, idesc, k);
    umma_commit(&bars[1]);
  }

  // delta = rowsum(dO * O) while the MMAs run (query row = tid)
  float delta = 0.f;
  {
    const long long off = (static_cast<long long>(b) * kS + tid) * p.H + h * kD;
    const uint4* o4 = reinterpret_cast<const uint4*>(p.ctx_in + off);
    // dO row read from global (also in smem, but swizzled; global read is simpler and cached)
    const uint4* d4 = reinterpret_cast<const uint4*>(
        reinterpret_cast<const __nv_bfloat16*>(p.ctx) + off);  // p.ctx aliases dctx in bwd
#pragma unroll
    for (int i = 0; i < kD / 8; ++i) {
      const uint4 a = o4[i];
      const uint4 g = d4[i];
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
      const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float2 x = unpack_bf16x2(aw[t]);
        const float2 y = unpack_bf16x2(gw[t]);
        delta += x.x * y.x + x.y * y.y;
      }
    }
  }
  const float lse = p.lse[static_cast<long long>(bh) * kS + tid];

  mbar_wait(&bars[1], 0);
  tcgen05_fence_after();

  const uint32_t trow = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
  const float sc = p.scale * kLog2e;
  const bool has_dropout = p.dropout_p > 0.f;
  uint64_t seed = 0;
  uint32_t thr16 = 0;
  float dscale = 1.f;
  if (has_dropout) {
    seed = dropout_seed(p.rng_state, p.rng_stream);
    thr16 = static_cast<uint32_t>(p.dropout_p * 65536.f);
    dscale = 1.f / (1.f - p.dropout_p);
  }
  const uint64_t drop_row = (static_cast<uint64_t>(bh) * kS + tid) * kS;
#pragma unroll 1
  for (int c = 0; c < 8; ++c) {  // 16 keys per step
    uint32_t vs[16], vd[16];
    tmem_ld_32x32b_x16(trow + cS + c * 16, vs);
    tmem_ld_32x32b_x16(trow + cdP + c * 16, vd);
    tmem_ld_wait();
    float pd[16], ds[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      pd[j] = exp2f(__uint_as_float(vs[j]) * sc + sMask[c * 16 + j] - lse);
      ds[j] = __uint_as_float(vd[j]);
    }
    if (has_dropout) {
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const uint32_t m = dropout_keep4(seed, (drop_row + c * 16 + j) >> 2, thr16);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const bool keep = (m >> t) & 1u;
          const float pj = pd[j + t];
          // dS uses the un-dropped P; the dropped/scaled P feeds dV
          ds[j + t] = pj * ((keep ? ds[j + t] * dscale : 0.f) - delta) * p.scale;
          pd[j + t] = keep ? pj * dscale : 0.f;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) ds[j] = pd[j] * (ds[j] - delta) * p.scale;
    }
    uint8_t* bp = (c >> 2) ? sP1 : sP0;
    uint8_t* bd = sdS + (c >> 2) * kTile;
#pragma unroll
    for (int j = 0; j < 16; j += 8) {
      const uint32_t off = sw128_offset(tid, (c & 3) * 16 + j);
      uint4 pk;
      pk.x = pack_bf16x2(pd[j], pd[j + 1]);
      pk.y = pack_bf16x2(pd[j + 2], pd[j + 3]);
      pk.z = pack_bf16x2(pd[j + 4], pd[j + 5]);
      pk.w = pack_bf16x2(pd[j + 6], pd[j + 7]);
      *reinterpret_cast<uint4*>(bp + off) = pk;
      pk.x = pack_bf16x2(ds[j], ds[j + 1]);
      pk.y = pack_bf16x2(ds[j + 2], ds[j + 3]);
      pk.z = pack_bf16x2(ds[j + 4], ds[j + 5]);
      pk.w = pack_bf16x2(ds[j + 6], ds[j + 7]);
      *reinterpret_cast<uint4*>(bd + off) = pk;
    }
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();

  if (warp == 0 && elect_one_sync()) {
    tcgen05_fence_after();
    // dV[key, d] = sum_q P[q,key] dO[q,d] : A = P (MN-major, 2 key-chunks 16KB apart), B = dO (MN)
    // dK[key, d] = sum_q dS[q,key] Q[q,d] : A = dS (MN-major),                         B = Q  (MN)
    constexpr uint32_t idesc_t = make_idesc_bf16_f32(128, 64, true, true);
#pragma unroll
    for (int j = 0; j < kS / 16; ++j) {
      const uint64_t da = make_smem_desc_sw128(smem_u32(sP0) + j * 2048, 2 * kTile, 1024);
      const uint64_t db = make_smem_desc_sw128(smem_u32(sdO) + j * 2048, kTile, 1024);
      umma_bf16_ss(tmem_base + cdV, da, db, idesc_t, j);
    }
#pragma unroll
    for (int j = 0; j < kS / 16; ++j) {
      const uint64_t da = make_smem_desc_sw128(smem_u32(sdS) + j * 2048, kTile, 1024);
      const uint64_t db = make_smem_desc_sw128(smem_u32(sQ) + j * 2048, kTile, 1024);
      umma_bf16_ss(tmem_base + cdK, da, db, idesc_t, j);
    }
    // dQ[q, d] = sum_key dS[q,key] K[key,d] : A = dS (K-major, 2 K-blocks), B = K (MN-major)
    constexpr uint32_t idesc_q = make_idesc_bf16_f32(128, 64, false, true);
#pragma unroll
    for (int j = 0; j < kS / 16; ++j) {
      const uint64_t da =
          make_smem_desc_sw128(smem_u32(sdS + (j >> 2) * kTile) + (j & 3) * 32, 16, 1024);
      const uint64_t db = make_smem_desc_sw128(smem_u32(sK) + j * 2048, kTile, 1024);
      umma_bf16_ss(tmem_base + cdQ, da, db, idesc_q, j);
    }
    umma_commit(&bars[2]);
  }
  mbar_wait(&bars[2], 0);
  tcgen05_fence_after();

  __nv_bfloat16* grow = p.dqkv + (static_cast<long long>(b) * kS + tid) * (3 * p.H) + h * kD;
  const uint32_t cols[3] = {cdQ, cdK, cdV};
#pragma unroll 1
  for (int t = 0; t < 3; ++t) {
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(trow + cols[t] + c * 32, v);
      tmem_ld_wait();
      __nv_bfloat16* o = grow + t * p.H + c * 32;
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 pk;
        pk.x = pack_bf16x2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
        pk.y = pack_bf16x2(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        pk.z = pack_bf16x2(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5]));
        pk.w = pack_bf16x2(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7]));
        *reinterpret_cast<uint4*>(o + j) = pk;
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

}  // namespace

// S = 128 with head_dim = 64 runs the single-tile kernels of this file; every other shape (and
// S = 128 when SKY_ATTN_TILED=1, for A/B comparisons) the flash-style tiled kernels of
// attention_tiled_sm100.cu, which also reject (930) what no kernel supports
static bool force_tiled() {
  static int v = -1;
  if (v < 0) {
    const char* e = std::getenv("SKY_ATTN_TILED");
    v = (e != nullptr && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

int launch_attention_fwd(const AttnArgs& a, cudaStream_t stream) {
  if (a.head_dim != kD || a.S != kS || force_tiled()) return launch_attention_fwd_tiled(a, stream);
  if (a.dropout_p > 0.f && a.rng_state == nullptr) return 903;
  const int H = a.heads * kD;
  CUtensorMap tm;
  int rc = make_tmap_bf16_2d(&tm, a.qkv, 3ull * H, static_cast<uint64_t>(a.B) * kS, 3ull * H, 64,
                             128);
  if (rc) return rc;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attention_fwd_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdSmem);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr = true;
  }
  AttnDev d;
  d.mask = a.mask;
  d.ctx = reinterpret_cast<__nv_bfloat16*>(a.ctx);
  d.lse = a.lse;
  d.ctx_in = nullptr;
  d.dqkv = nullptr;
  d.heads = a.heads;
  d.H = H;
  d.scale = a.scale;
  d.dropout_p = a.dropout_p;
  d.rng_state = a.rng_state;
  d.rng_stream = a.rng_stream;
  cudaError_t le = launch_pdl(attention_fwd_kernel, dim3(a.B * a.heads), dim3(128), kFwdSmem, stream, tm, d);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}

int launch_attention_bwd(const AttnArgs& a, cudaStream_t stream) {
  if (a.head_dim != kD || a.S != kS || force_tiled()) return launch_attention_bwd_tiled(a, stream);
  if (a.dropout_p > 0.f && a.rng_state == nullptr) return 903;
  if (a.lse == nullptr || a.ctx == nullptr || a.dctx == nullptr) return 931;
  const int H = a.heads * kD;
  CUtensorMap tm, tdo;
  int rc = make_tmap_bf16_2d(&tm, a.qkv, 3ull * H, static_cast<uint64_t>(a.B) * kS, 3ull * H, 64,
                             128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tdo, a.dctx, static_cast<uint64_t>(H), static_cast<uint64_t>(a.B) * kS,
                         static_cast<uint64_t>(H), 64, 128);
  if (rc) return rc;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attention_bwd_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdSmem);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr = true;
  }
  AttnDev d;
  d.mask = a.mask;
  // in the backward kernel `ctx` carries dctx (gradient wrt attention output) and `ctx_in` the
  // saved forward output
  d.ctx = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(a.dctx));
  d.ctx_in = reinterpret_cast<const __nv_bfloat16*>(a.ctx);
  d.lse = a.lse;
  d.dqkv = reinterpret_cast<__nv_bfloat16*>(a.dqkv);
  d.heads = a.heads;
  d.H = H;
  d.scale = a.scale;
  d.dropout_p = a.dropout_p;
  d.rng_state = a.rng_state;
  d.rng_stream = a.rng_stream;
  cudaError_t le = launch_pdl(attention_bwd_kernel, dim3(a.B * a.heads), dim3(128), kBwdSmem, stream, tm, tdo, d);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace sky
