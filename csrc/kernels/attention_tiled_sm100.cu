// Self-attention for ANY sequence length (S % 8 == 0) and head size (D % 8 == 0, 8 <= D <= 128) on
// tcgen05: flash-style tiling over 128-key blocks, so the native path covers everything the
// reference's eager attention does (scaelum/model/bert_layers.py:249-275 materialises
// [B, h, S, S] for any S <= 512 and any head size).  S = 128 with D = 64 keeps its specialised
// single-tile kernels (attention_sm100.cu); this file is the general case.
//
//   forward   one CTA per (batch, head, 128-query tile), loop over key tiles:
//               S = Q K_j^T (UMMA 128x128xD) -> TMEM -> online softmax in registers (running row
//               max m, row sum l, + additive mask, + dropout) -> P_j (bf16, swizzled smem) ->
//               O_j = P_j V_j (UMMA 128xDPx128) -> O = O * 2^(m_old - m_new) + O_j (in registers
//               for DP = 64; for DP = 128 O stays in TMEM: rescaled in place, then accumulated
//               into by the UMMA).  K / V tiles are double buffered: tile j+1 streams in while
//               tile j is processed.
//   backward  two kernels, both recompute P from the saved log-sum-exp:
//               dQ  : one CTA per query tile, loop over key tiles: dS_j -> dQ += dS_j K_j
//               dKV : one CTA per key tile, loop over query tiles: dV += P^T dO, dK += dS^T Q
//                     (accumulated in TMEM across the loop: S, dP, dV, dK = 256 + 2 DP columns)
//             no atomics, deterministic; the price is computing S and dP twice.
//
// Head sizes: the kernels are instantiated for a padded head size DP in {64, 128}, i.e. one or two
// SWIZZLE_128B K-blocks of 64 columns per operand tile.  D = 64 views the [B * S, C] activations
// through a 3D tensor map (column, position, batch); every other D through a 4D map (column,
// head section, position, batch) whose row is exactly D columns long, so the box columns past D
// arrive as zeros (which add nothing to Q K^T, dO V^T or dS K) and the padded output columns are
// never stored.  The 16-byte TMA stride rule on a row of D bf16 is where D % 8 == 0 comes from.
//
// Ragged tiles: rows past the end of a sequence arrive as zeros the same way; keys past S get an
// additive -1e30 (probability exactly 0), queries past S are computed on zeros and never stored.
// Dropout indexing is the same flat [B, heads, S, S] element index as the S = 128 kernels and the
// host replica (skycomputing_b200/ops/dropout_ref.py).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "api.h"
#include "launch_util.h"
#include "sm100_ptx.cuh"

namespace sky {

int make_tmap_bf16_3d(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t middle,
                      uint64_t outer, uint64_t ld_middle_elems, uint64_t ld_outer_elems,
                      uint32_t box_inner, uint32_t box_middle);
int make_tmap_bf16_4d(CUtensorMap* tm, const void* ptr, const uint64_t (&dims)[4],
                      const uint64_t (&ld_elems)[3], uint32_t box_inner, uint32_t box_third);

namespace {

constexpr int kT = 128;              // queries / keys per tile
constexpr int kD = 64;               // columns of one SWIZZLE_128B K-block (and the unpadded D)
constexpr int kTile = kT * kD * 2;   // 16 KB: one [128 x 64] bf16 tile
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kNegBig = -1.0e30f;  // additive mask of keys past the end of the sequence

__device__ __forceinline__ uint32_t sw128_offset(int row, int col) {
  const uint32_t chunk = static_cast<uint32_t>(col >> 3) ^ static_cast<uint32_t>(row & 7);
  return static_cast<uint32_t>(row) * 128u + (chunk << 4) + static_cast<uint32_t>(col & 7) * 2u;
}

struct AttnTDev {
  const float* mask;            // [B, S] additive or null
  __nv_bfloat16* ctx;           // fwd: output [B*S, H]
  float* lse;                   // [B*heads, S] log2-domain log-sum-exp
  const __nv_bfloat16* ctx_in;  // bwd: saved forward output
  const __nv_bfloat16* dctx;    // bwd: gradient of the attention output
  __nv_bfloat16* dqkv;          // bwd: [B*S, 3H]
  int S, heads, H, n_tiles;
  float scale, dropout_p;
  const uint64_t* rng_state;
  uint32_t rng_stream;
  int D;                        // head size (the padded kernels; D = 64 uses the constant)
};

// Template parameters of every kernel: DP = padded head size (64 or 128), kPad = the operands come
// through the 4D tensor map (any D but 64).  D = 64 is <64, false>.
template <bool kPad>
__device__ __forceinline__ int head_dim(const AttnTDev& p) {
  return kPad ? p.D : kD;
}

// One [128 rows x 64 columns] box of head h: column block `cb`, section `sec` of the row (qkv:
// 0 = Q, 1 = K, 2 = V; dO has a single section), rows row..row+127 of sequence b.
template <bool kPad>
__device__ __forceinline__ void load_box(void* dst, const CUtensorMap* tm, uint64_t* bar,
                                         const AttnTDev& p, int sec, int h, int cb, int row, int b) {
  if (kPad)
    tma_load_4d(dst, tm, bar, cb * kD, sec * p.heads + h, row, b);
  else
    tma_load_3d(dst, tm, bar, sec * p.H + h * kD, row, b);
}
template <int DP, bool kPad>
__device__ __forceinline__ void load_op(uint8_t* dst, const CUtensorMap* tm, uint64_t* bar,
                                        const AttnTDev& p, int sec, int h, int row, int b) {
#pragma unroll
  for (int cb = 0; cb < DP / kD; ++cb)
    load_box<kPad>(dst + cb * kTile, tm, bar, p, sec, h, cb, row, b);
}

// S (or dP) = A B^T over the head dimension: both operands K-major, DP / 64 K-blocks; only the
// k-steps that hold real columns are issued
template <int DP, bool kPad>
__device__ __forceinline__ void umma_over_head(uint32_t tmem_d, const uint8_t* sA, const uint8_t* sB,
                                               int D) {
  constexpr uint32_t idesc = make_idesc_bf16_f32(128, 128, false, false);
  const uint64_t da = make_smem_desc_sw128(smem_u32(sA), 16, 1024);
  const uint64_t db = make_smem_desc_sw128(smem_u32(sB), 16, 1024);
  const int nk = kPad ? (D + 15) / 16 : kD / 16;
#pragma unroll
  for (int k = 0; k < nk; ++k) {
    const uint64_t off = (k >> 2) * (kTile >> 4) + 2 * (k & 3);
    umma_bf16_ss(tmem_d, da + off, db + off, idesc, k);
  }
}

// the first `ncols` (a multiple of 8) of a 64-column row
__device__ __forceinline__ void store_row64(__nv_bfloat16* dst, const float (&o)[64], float mul,
                                            int ncols) {
#pragma unroll
  for (int j = 0; j < 64; j += 8) {
    if (j >= ncols) break;
    uint4 pk;
    pk.x = pack_bf16x2(o[j] * mul, o[j + 1] * mul);
    pk.y = pack_bf16x2(o[j + 2] * mul, o[j + 3] * mul);
    pk.z = pack_bf16x2(o[j + 4] * mul, o[j + 5] * mul);
    pk.w = pack_bf16x2(o[j + 6] * mul, o[j + 7] * mul);
    *reinterpret_cast<uint4*>(dst + j) = pk;
  }
}

// the first `ncols` (a multiple of 8) fp32 columns of a TMEM row as bf16; tcgen05.ld is
// warp-collective, so every lane loads and only lanes with `store` write
__device__ __forceinline__ void store_tmem_row(__nv_bfloat16* dst, uint32_t taddr, int ncols,
                                               float mul, bool store) {
#pragma unroll 1
  for (int c0 = 0; c0 < ncols; c0 += 32) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(taddr + c0, v);
    tmem_ld_wait();
    if (!store) continue;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      if (c0 + j >= ncols) break;
      uint4 pk;
      pk.x = pack_bf16x2(__uint_as_float(v[j]) * mul, __uint_as_float(v[j + 1]) * mul);
      pk.y = pack_bf16x2(__uint_as_float(v[j + 2]) * mul, __uint_as_float(v[j + 3]) * mul);
      pk.z = pack_bf16x2(__uint_as_float(v[j + 4]) * mul, __uint_as_float(v[j + 5]) * mul);
      pk.w = pack_bf16x2(__uint_as_float(v[j + 6]) * mul, __uint_as_float(v[j + 7]) * mul);
      *reinterpret_cast<uint4*>(dst + c0 + j) = pk;
    }
  }
}

// ----------------------------------------------------------------------------------------------
// forward
// ----------------------------------------------------------------------------------------------
// Q, 2 x (K, V), P (2 blocks), mask, barriers
template <int DP>
constexpr int fwd_smem() { return 5 * (DP / kD) * kTile + 2 * kTile + 512 + 128 + 1024; }

template <int DP, bool kPad>
__global__ void __launch_bounds__(128, 1)
attention_fwd_tiled_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnTDev p) {
  constexpr int kOp = (DP / kD) * kTile;   // one [128 x DP] operand tile
  constexpr bool kOTmem = DP > 64;         // O accumulated in TMEM (o_acc[128] would spill)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + kOp;        // [2 buffers][K, V]
  uint8_t* sP = smem + 5 * kOp;     // two [128 x 64] K-blocks
  float* sMask = reinterpret_cast<float*>(smem + 5 * kOp + 2 * kTile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 5 * kOp + 2 * kTile + 512);
  uint64_t* bar_q = &bars[0];
  uint64_t* bar_kv = &bars[1];      // [2]
  uint64_t* bar_s = &bars[3];
  uint64_t* bar_o = &bars[4];
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int qt = blockIdx.x % p.n_tiles;
  const int bh = blockIdx.x / p.n_tiles;
  const int b = bh / p.heads;
  const int h = bh % p.heads;
  const int q = qt * kT + tid;      // my query position
  const bool q_ok = q < p.S;
  const int D = head_dim<kPad>(p);

  if (tid == 0) {
    tma_prefetch_desc(&tmap_qkv);
    for (int i = 0; i < 5; ++i) mbar_init(&bars[i], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, 256);
    tmem_relinquish();
  }
  pdl_wait();
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t trow = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);

  const bool issuer = warp == 0 && elect_one_sync();
  if (issuer) {
    mbar_expect_tx(bar_q, kOp);
    load_op<DP, kPad>(sQ, &tmap_qkv, bar_q, p, 0, h, qt * kT, b);
    mbar_expect_tx(&bar_kv[0], 2 * kOp);
    load_op<DP, kPad>(sKV, &tmap_qkv, &bar_kv[0], p, 1, h, 0, b);
    load_op<DP, kPad>(sKV + kOp, &tmap_qkv, &bar_kv[0], p, 2, h, 0, b);
  }

  const float sc = p.scale * kLog2e;
  const bool has_dropout = p.dropout_p > 0.f;
  uint64_t seed = 0;
  uint32_t thr16 = 0;
  if (has_dropout) {
    seed = dropout_seed(p.rng_state, p.rng_stream);
    thr16 = static_cast<uint32_t>(p.dropout_p * 65536.f);
  }
  const uint64_t drop_row = (static_cast<uint64_t>(bh) * p.S + (q_ok ? q : 0)) * p.S;

  float o_acc[kOTmem ? 1 : 64];
  if constexpr (!kOTmem) {
#pragma unroll
    for (int j = 0; j < 64; ++j) o_acc[j] = 0.f;
  }
  float m_run = -INFINITY, l_run = 0.f;

  for (int j = 0; j < p.n_tiles; ++j) {
    const int buf = j & 1;
    uint8_t* sK = sKV + buf * 2 * kOp;
    uint8_t* sV = sK + kOp;
    // additive mask of this key tile (log2 domain); keys past the sequence end get -1e30
    {
      const int k = j * kT + tid;
      sMask[tid] = k < p.S ? (p.mask ? p.mask[b * p.S + k] * kLog2e : 0.f) : kNegBig;
    }
    if (issuer) {
      if (j + 1 < p.n_tiles) {   // the other buffer's tile (j - 1) is fully consumed: prefetch
        uint8_t* nK = sKV + (buf ^ 1) * 2 * kOp;
        mbar_expect_tx(&bar_kv[buf ^ 1], 2 * kOp);
        load_op<DP, kPad>(nK, &tmap_qkv, &bar_kv[buf ^ 1], p, 1, h, (j + 1) * kT, b);
        load_op<DP, kPad>(nK + kOp, &tmap_qkv, &bar_kv[buf ^ 1], p, 2, h, (j + 1) * kT, b);
      }
      if (j == 0) mbar_wait(bar_q, 0);
      mbar_wait(&bar_kv[buf], (j >> 1) & 1);
      tcgen05_fence_after();
      umma_over_head<DP, kPad>(tmem_base, sQ, sK, D);
      umma_commit(bar_s);
    }
    __syncthreads();             // sMask visible
    mbar_wait(bar_s, j & 1);
    tcgen05_fence_after();

    // ---- online softmax over my row ----
    float mx = m_run;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(trow + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int t = 0; t < 32; ++t) mx = fmaxf(mx, __uint_as_float(v[t]) * sc + sMask[c * 32 + t]);
    }
    const float alpha = exp2f(m_run - mx);   // 0 on the first tile (m_run = -inf, mx finite)
    float sum = 0.f;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(trow + c * 32, v);
      tmem_ld_wait();
      float e[32];
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        e[t] = exp2f(__uint_as_float(v[t]) * sc + sMask[c * 32 + t] - mx);
        sum += e[t];
      }
      if (has_dropout) {
#pragma unroll
        for (int t = 0; t < 32; t += 4) {
          const uint32_t m =
              dropout_keep4(seed, (drop_row + static_cast<uint64_t>(j * kT + c * 32 + t)) >> 2, thr16);
          e[t] = (m & 1u) ? e[t] : 0.f;
          e[t + 1] = (m & 2u) ? e[t + 1] : 0.f;
          e[t + 2] = (m & 4u) ? e[t + 2] : 0.f;
          e[t + 3] = (m & 8u) ? e[t + 3] : 0.f;
        }
      }
      uint8_t* blk = sP + (c >> 1) * kTile;
#pragma unroll
      for (int t = 0; t < 32; t += 8) {
        uint4 pk;
        pk.x = pack_bf16x2(e[t], e[t + 1]);
        pk.y = pack_bf16x2(e[t + 2], e[t + 3]);
        pk.z = pack_bf16x2(e[t + 4], e[t + 5]);
        pk.w = pack_bf16x2(e[t + 6], e[t + 7]);
        *reinterpret_cast<uint4*>(blk + sw128_offset(tid, (c & 1) * 32 + t)) = pk;
      }
    }
    l_run = l_run * alpha + sum;
    m_run = mx;
    if (kOTmem && j > 0) {   // O *= alpha in place; the P V UMMA below then accumulates into it
#pragma unroll 1
      for (int c = 0; c < D; c += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(trow + 128 + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int t = 0; t < 32; ++t) v[t] = __float_as_uint(__uint_as_float(v[t]) * alpha);
        tmem_st_32x32b_x32(trow + 128 + c, v);
      }
      tmem_st_wait();
    }
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();

    if (issuer) {
      tcgen05_fence_after();
      constexpr uint32_t idesc = make_idesc_bf16_f32(128, DP, false, true);
#pragma unroll
      for (int k = 0; k < kT / 16; ++k) {
        const uint64_t da =
            make_smem_desc_sw128(smem_u32(sP + (k >> 2) * kTile) + (k & 3) * 32, 16, 1024);
        const uint64_t db = make_smem_desc_sw128(smem_u32(sV) + k * 2048, kTile, 1024);
        umma_bf16_ss(tmem_base + 128, da, db, idesc, kOTmem ? (j > 0 || k > 0) : k);
      }
      umma_commit(bar_o);
    }
    mbar_wait(bar_o, j & 1);
    tcgen05_fence_after();
    if constexpr (!kOTmem) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {   // fully unrolled: o_acc must stay in registers
        uint32_t v[32];
        tmem_ld_32x32b_x32(trow + 128 + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int t = 0; t < 32; ++t)
          o_acc[c * 32 + t] = fmaf(o_acc[c * 32 + t], alpha, __uint_as_float(v[t]));
      }
    }
    tcgen05_fence_before();
  }

  if constexpr (kOTmem) {
    const float inv = (has_dropout ? 1.f / (1.f - p.dropout_p) : 1.f) / l_run;
    tcgen05_fence_after();
    store_tmem_row(p.ctx + (static_cast<long long>(b) * p.S + (q_ok ? q : 0)) * p.H + h * D,
                   trow + 128, D, inv, q_ok);
    if (q_ok && p.lse != nullptr) p.lse[static_cast<long long>(bh) * p.S + q] = m_run + log2f(l_run);
    tcgen05_fence_before();
  } else if (q_ok) {
    const float inv = (has_dropout ? 1.f / (1.f - p.dropout_p) : 1.f) / l_run;
    store_row64(p.ctx + (static_cast<long long>(b) * p.S + q) * p.H + h * D, o_acc, inv, D);
    if (p.lse != nullptr) p.lse[static_cast<long long>(bh) * p.S + q] = m_run + log2f(l_run);
  }
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ----------------------------------------------------------------------------------------------
// backward: shared pieces
// ----------------------------------------------------------------------------------------------
// P and dS of one [128 queries x 128 keys] tile from S and dP in TMEM (columns 0..127 / 128..255):
// P = 2^(s * sc + mask - lse), dS = P * (dP * keep / (1-p) - delta) * scale; the dropped / scaled
// P (-> dV) goes to sP, dS to sdS, both as two swizzled [128 x 64] K-blocks indexed [query][key].
struct BwdRow {
  float lse, delta;
  uint64_t drop_row;
};

__device__ __forceinline__ void softmax_bwd_tile(uint32_t trow, const float* sMask, const BwdRow& r,
                                                 int key0, float sc, float scale, bool has_dropout,
                                                 uint64_t seed, uint32_t thr16, float dscale,
                                                 int tid, uint8_t* sP, uint8_t* sdS) {
#pragma unroll 1
  for (int c = 0; c < 8; ++c) {   // 16 keys per step
    uint32_t vs[16], vd[16];
    tmem_ld_32x32b_x16(trow + c * 16, vs);
    tmem_ld_32x32b_x16(trow + 128 + c * 16, vd);
    tmem_ld_wait();
    float pd[16], ds[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      pd[t] = exp2f(__uint_as_float(vs[t]) * sc + sMask[c * 16 + t] - r.lse);
      ds[t] = __uint_as_float(vd[t]);
    }
    if (has_dropout) {
#pragma unroll
      for (int t = 0; t < 16; t += 4) {
        const uint32_t m =
            dropout_keep4(seed, (r.drop_row + static_cast<uint64_t>(key0 + c * 16 + t)) >> 2, thr16);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool keep = (m >> u) & 1u;
          const float pj = pd[t + u];
          ds[t + u] = pj * ((keep ? ds[t + u] * dscale : 0.f) - r.delta) * scale;
          pd[t + u] = keep ? pj * dscale : 0.f;
        }
      }
    } else {
#pragma unroll
      for (int t = 0; t < 16; ++t) ds[t] = pd[t] * (ds[t] - r.delta) * scale;
    }
    uint8_t* bp = sP != nullptr ? sP + (c >> 2) * kTile : nullptr;
    uint8_t* bd = sdS + (c >> 2) * kTile;
#pragma unroll
    for (int t = 0; t < 16; t += 8) {
      const uint32_t off = sw128_offset(tid, (c & 3) * 16 + t);
      uint4 pk;
      if (bp != nullptr) {
        pk.x = pack_bf16x2(pd[t], pd[t + 1]);
        pk.y = pack_bf16x2(pd[t + 2], pd[t + 3]);
        pk.z = pack_bf16x2(pd[t + 4], pd[t + 5]);
        pk.w = pack_bf16x2(pd[t + 6], pd[t + 7]);
        *reinterpret_cast<uint4*>(bp + off) = pk;
      }
      pk.x = pack_bf16x2(ds[t], ds[t + 1]);
      pk.y = pack_bf16x2(ds[t + 2], ds[t + 3]);
      pk.z = pack_bf16x2(ds[t + 4], ds[t + 5]);
      pk.w = pack_bf16x2(ds[t + 6], ds[t + 7]);
      *reinterpret_cast<uint4*>(bd + off) = pk;
    }
  }
}

// lse and delta = rowsum(dO * O) of query `q` (zeros / +big for rows past the sequence end, which
// makes P and dS of such rows exactly 0)
template <bool kPad>
__device__ __forceinline__ BwdRow load_bwd_row(const AttnTDev& p, int b, int h, int bh, int q) {
  BwdRow r;
  if (q >= p.S) {
    r.lse = 1.0e30f;
    r.delta = 0.f;
    r.drop_row = 0;
    return r;
  }
  const int D = head_dim<kPad>(p);
  const long long off = (static_cast<long long>(b) * p.S + q) * p.H + h * D;
  const uint4* o4 = reinterpret_cast<const uint4*>(p.ctx_in + off);
  const uint4* d4 = reinterpret_cast<const uint4*>(p.dctx + off);
  float delta = 0.f;
#pragma unroll
  for (int i = 0; i < D / 8; ++i) {
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
  r.delta = delta;
  r.lse = p.lse[static_cast<long long>(bh) * p.S + q];
  r.drop_row = (static_cast<uint64_t>(bh) * p.S + q) * p.S;
  return r;
}

// ----------------------------------------------------------------------------------------------
// backward: dQ (one CTA per query tile, loop over key tiles)
// ----------------------------------------------------------------------------------------------
// Q, dO, K, V, dS (2 blocks)
template <int DP>
constexpr int bwd_q_smem() { return 4 * (DP / kD) * kTile + 2 * kTile + 512 + 128 + 1024; }

template <int DP, bool kPad>
__global__ void __launch_bounds__(128, 1)
attention_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmap_qkv,
                        const __grid_constant__ CUtensorMap tmap_do, const AttnTDev p) {
  constexpr int kOp = (DP / kD) * kTile;
  // DP = 128: dQ accumulates in TMEM columns 256..383 (dq[128] would spill); DP = 64: in registers
  constexpr bool kQTmem = DP > 64;
  constexpr uint32_t kCols = kQTmem ? 512 : 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;
  uint8_t* sdO = smem + kOp;
  uint8_t* sK = smem + 2 * kOp;
  uint8_t* sV = smem + 3 * kOp;
  uint8_t* sdS = smem + 4 * kOp;
  float* sMask = reinterpret_cast<float*>(smem + 4 * kOp + 2 * kTile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 4 * kOp + 2 * kTile + 512);
  uint64_t* bar_q = &bars[0];
  uint64_t* bar_kv = &bars[1];
  uint64_t* bar_s = &bars[2];
  uint64_t* bar_o = &bars[3];
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int qt = blockIdx.x % p.n_tiles;
  const int bh = blockIdx.x / p.n_tiles;
  const int b = bh / p.heads;
  const int h = bh % p.heads;
  const int q = qt * kT + tid;
  const int D = head_dim<kPad>(p);

  if (tid == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, kCols);
    tmem_relinquish();
  }
  pdl_wait();
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t trow = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
  const bool issuer = warp == 0 && elect_one_sync();
  if (issuer) {
    mbar_expect_tx(bar_q, 2 * kOp);
    load_op<DP, kPad>(sQ, &tmap_qkv, bar_q, p, 0, h, qt * kT, b);
    load_op<DP, kPad>(sdO, &tmap_do, bar_q, p, 0, h, qt * kT, b);
  }
  const BwdRow row = load_bwd_row<kPad>(p, b, h, bh, q);
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
  float dq[kQTmem ? 1 : 64];
  if constexpr (!kQTmem) {
#pragma unroll
    for (int j = 0; j < 64; ++j) dq[j] = 0.f;
  }

  for (int j = 0; j < p.n_tiles; ++j) {
    {
      const int k = j * kT + tid;
      sMask[tid] = k < p.S ? (p.mask ? p.mask[b * p.S + k] * kLog2e : 0.f) : kNegBig;
    }
    if (issuer) {
      mbar_expect_tx(bar_kv, 2 * kOp);
      load_op<DP, kPad>(sK, &tmap_qkv, bar_kv, p, 1, h, j * kT, b);
      load_op<DP, kPad>(sV, &tmap_qkv, bar_kv, p, 2, h, j * kT, b);
      if (j == 0) mbar_wait(bar_q, 0);
      mbar_wait(bar_kv, j & 1);
      tcgen05_fence_after();
      umma_over_head<DP, kPad>(tmem_base, sQ, sK, D);
      umma_over_head<DP, kPad>(tmem_base + 128, sdO, sV, D);
      umma_commit(bar_s);
    }
    __syncthreads();
    mbar_wait(bar_s, j & 1);
    tcgen05_fence_after();
    softmax_bwd_tile(trow, sMask, row, j * kT, sc, p.scale, has_dropout, seed, thr16, dscale, tid,
                     nullptr, sdS);
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    if (issuer) {
      tcgen05_fence_after();
      // dQ_j[q, d] = sum_key dS[q, key] K[key, d]: A = dS (K-major, 2 K-blocks), B = K (MN-major)
      constexpr uint32_t idesc_q = make_idesc_bf16_f32(128, DP, false, true);
#pragma unroll
      for (int k = 0; k < kT / 16; ++k) {
        const uint64_t da =
            make_smem_desc_sw128(smem_u32(sdS + (k >> 2) * kTile) + (k & 3) * 32, 16, 1024);
        const uint64_t db = make_smem_desc_sw128(smem_u32(sK) + k * 2048, kTile, 1024);
        if constexpr (kQTmem)
          umma_bf16_ss(tmem_base + 256, da, db, idesc_q, (j > 0 || k > 0) ? 1u : 0u);
        else
          umma_bf16_ss(tmem_base, da, db, idesc_q, k);   // S is dead: its columns take dQ_j
      }
      umma_commit(bar_o);
    }
    mbar_wait(bar_o, j & 1);
    tcgen05_fence_after();
    if constexpr (!kQTmem) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {   // fully unrolled: dq must stay in registers
        uint32_t v[32];
        tmem_ld_32x32b_x32(trow + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int t = 0; t < 32; ++t) dq[c * 32 + t] += __uint_as_float(v[t]);
      }
    }
    tcgen05_fence_before();
    __syncthreads();   // everybody has read dQ_j (and K / V): the next tile may overwrite them
  }
  if constexpr (kQTmem) {
    tcgen05_fence_after();
    store_tmem_row(p.dqkv + (static_cast<long long>(b) * p.S + (q < p.S ? q : 0)) * (3 * p.H) + h * D,
                   trow + 256, D, 1.f, q < p.S);
    tcgen05_fence_before();
  } else if (q < p.S) {
    store_row64(p.dqkv + (static_cast<long long>(b) * p.S + q) * (3 * p.H) + h * D, dq, 1.f, D);
  }
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, kCols);
  }
}

// ----------------------------------------------------------------------------------------------
// backward: dK, dV (one CTA per key tile, loop over query tiles, accumulators stay in TMEM)
// ----------------------------------------------------------------------------------------------
// K, V, Q, dO, P (2), dS (2)
template <int DP>
constexpr int bwd_kv_smem() { return 4 * (DP / kD) * kTile + 4 * kTile + 512 + 128 + 1024; }

template <int DP, bool kPad>
__global__ void __launch_bounds__(128, 1)
attention_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tmap_qkv,
                         const __grid_constant__ CUtensorMap tmap_do, const AttnTDev p) {
  constexpr int kOp = (DP / kD) * kTile;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sK = smem;
  uint8_t* sV = smem + kOp;
  uint8_t* sQ = smem + 2 * kOp;
  uint8_t* sdO = smem + 3 * kOp;
  uint8_t* sP = smem + 4 * kOp;
  uint8_t* sdS = smem + 4 * kOp + 2 * kTile;
  float* sMask = reinterpret_cast<float*>(smem + 4 * kOp + 4 * kTile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 4 * kOp + 4 * kTile + 512);
  uint64_t* bar_kv = &bars[0];
  uint64_t* bar_q = &bars[1];
  uint64_t* bar_s = &bars[2];
  uint64_t* bar_o = &bars[3];
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int kt = blockIdx.x % p.n_tiles;
  const int bh = blockIdx.x / p.n_tiles;
  const int b = bh / p.heads;
  const int h = bh % p.heads;
  const int D = head_dim<kPad>(p);
  constexpr uint32_t cdV = 256, cdK = 256 + DP;   // DP = 128: exactly the 512 columns

  if (tid == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, 512);
    tmem_relinquish();
  }
  pdl_wait();
  pdl_launch_dependents();
  {
    const int k = kt * kT + tid;
    sMask[tid] = k < p.S ? (p.mask ? p.mask[b * p.S + k] * kLog2e : 0.f) : kNegBig;
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t trow = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
  const bool issuer = warp == 0 && elect_one_sync();
  if (issuer) {
    mbar_expect_tx(bar_kv, 2 * kOp);
    load_op<DP, kPad>(sK, &tmap_qkv, bar_kv, p, 1, h, kt * kT, b);
    load_op<DP, kPad>(sV, &tmap_qkv, bar_kv, p, 2, h, kt * kT, b);
  }
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

  for (int i = 0; i < p.n_tiles; ++i) {
    if (issuer) {
      mbar_expect_tx(bar_q, 2 * kOp);
      load_op<DP, kPad>(sQ, &tmap_qkv, bar_q, p, 0, h, i * kT, b);
      load_op<DP, kPad>(sdO, &tmap_do, bar_q, p, 0, h, i * kT, b);
    }
    const BwdRow row = load_bwd_row<kPad>(p, b, h, bh, i * kT + tid);   // overlaps the loads
    if (issuer) {
      if (i == 0) mbar_wait(bar_kv, 0);
      mbar_wait(bar_q, i & 1);
      tcgen05_fence_after();
      umma_over_head<DP, kPad>(tmem_base, sQ, sK, D);
      umma_over_head<DP, kPad>(tmem_base + 128, sdO, sV, D);
      umma_commit(bar_s);
    }
    mbar_wait(bar_s, i & 1);
    tcgen05_fence_after();
    softmax_bwd_tile(trow, sMask, row, kt * kT, sc, p.scale, has_dropout, seed, thr16, dscale, tid,
                     sP, sdS);
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    if (issuer) {
      tcgen05_fence_after();
      // dV[key, d] += sum_q P[q, key] dO[q, d]; dK[key, d] += sum_q dS[q, key] Q[q, d]:
      // A = P / dS read MN-major (key-chunks one tile apart), B = dO / Q (MN-major, DP / 64
      // column blocks one tile apart)
      constexpr uint32_t idesc_t = make_idesc_bf16_f32(128, DP, true, true);
#pragma unroll
      for (int k = 0; k < kT / 16; ++k) {
        const uint64_t da = make_smem_desc_sw128(smem_u32(sP) + k * 2048, kTile, 1024);
        const uint64_t db = make_smem_desc_sw128(smem_u32(sdO) + k * 2048, kTile, 1024);
        umma_bf16_ss(tmem_base + cdV, da, db, idesc_t, (i > 0 || k > 0) ? 1u : 0u);
      }
#pragma unroll
      for (int k = 0; k < kT / 16; ++k) {
        const uint64_t da = make_smem_desc_sw128(smem_u32(sdS) + k * 2048, kTile, 1024);
        const uint64_t db = make_smem_desc_sw128(smem_u32(sQ) + k * 2048, kTile, 1024);
        umma_bf16_ss(tmem_base + cdK, da, db, idesc_t, (i > 0 || k > 0) ? 1u : 0u);
      }
      umma_commit(bar_o);
    }
    // Q / dO / P / dS are read by these MMAs: the next query tile may only overwrite them once
    // they have retired
    mbar_wait(bar_o, i & 1);
    tcgen05_fence_after();
    tcgen05_fence_before();
    __syncthreads();
  }

  tcgen05_fence_after();
  const int key = kt * kT + tid;
  {
    // tcgen05.ld is warp-collective (.sync.aligned): every lane loads, only rows of real keys store
    __nv_bfloat16* grow =
        p.dqkv + (static_cast<long long>(b) * p.S + (key < p.S ? key : 0)) * (3 * p.H) + h * D;
    if constexpr (DP > 64) {
      store_tmem_row(grow + p.H, trow + cdK, D, 1.f, key < p.S);
      store_tmem_row(grow + 2 * p.H, trow + cdV, D, 1.f, key < p.S);
    } else {
#pragma unroll
      for (int t = 0; t < 2; ++t) {   // t = 0: dK -> K section, t = 1: dV -> V section
        float o[64];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(trow + (t == 0 ? cdK : cdV) + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 32; ++u) o[c * 32 + u] = __uint_as_float(v[u]);
        }
        if (key < p.S) store_row64(grow + (t + 1) * p.H, o, 1.f, D);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int fill_dev(const AttnArgs& a, AttnTDev* d) {
  if (!attention_supported(a.S, a.head_dim)) return 930;
  if (a.dropout_p > 0.f && a.rng_state == nullptr) return 903;
  d->mask = a.mask;
  d->ctx = reinterpret_cast<__nv_bfloat16*>(a.ctx);
  d->lse = a.lse;
  d->ctx_in = reinterpret_cast<const __nv_bfloat16*>(a.ctx);
  d->dctx = reinterpret_cast<const __nv_bfloat16*>(a.dctx);
  d->dqkv = reinterpret_cast<__nv_bfloat16*>(a.dqkv);
  d->S = a.S;
  d->heads = a.heads;
  d->H = a.heads * a.head_dim;
  d->n_tiles = (a.S + kT - 1) / kT;
  d->scale = a.scale;
  d->dropout_p = a.dropout_p;
  d->rng_state = a.rng_state;
  d->rng_stream = a.rng_stream;
  d->D = a.head_dim;
  return 0;
}

// [B * S, sections * D] activations of `sections` head-sized column sections: a 3D map for D = 64,
// the padded 4D map otherwise (see the file comment); boxes are [128 rows x 64 columns]
int make_head_tmap(CUtensorMap* tm, const void* ptr, bool pad, int D, int sections, int S, int B) {
  const uint64_t C = static_cast<uint64_t>(sections) * D;
  if (!pad) return make_tmap_bf16_3d(tm, ptr, C, S, B, C, C * S, kD, kT);
  const uint64_t dims[4] = {static_cast<uint64_t>(D), static_cast<uint64_t>(sections),
                            static_cast<uint64_t>(S), static_cast<uint64_t>(B)};
  const uint64_t ld[3] = {static_cast<uint64_t>(D), C, C * S};
  return make_tmap_bf16_4d(tm, ptr, dims, ld, kD, kT);
}

template <class K>
int set_smem(K kern, int bytes, bool* done) {
  if (*done) return 0;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return static_cast<int>(e);
  *done = true;
  return 0;
}

template <int DP, bool kPad>
int launch_fwd(const AttnArgs& a, const AttnTDev& d, cudaStream_t stream) {
  CUtensorMap tm;
  int rc = make_head_tmap(&tm, a.qkv, kPad, a.head_dim, 3 * a.heads, a.S, a.B);
  if (rc) return rc;
  static bool attr = false;
  rc = set_smem(attention_fwd_tiled_kernel<DP, kPad>, fwd_smem<DP>(), &attr);
  if (rc) return rc;
  cudaError_t le = launch_pdl(attention_fwd_tiled_kernel<DP, kPad>, dim3(a.B * a.heads * d.n_tiles),
                              dim3(128), fwd_smem<DP>(), stream, tm, d);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}

template <int DP, bool kPad>
int launch_bwd(const AttnArgs& a, const AttnTDev& d, cudaStream_t stream) {
  CUtensorMap tm, tdo;
  int rc = make_head_tmap(&tm, a.qkv, kPad, a.head_dim, 3 * a.heads, a.S, a.B);
  if (rc) return rc;
  rc = make_head_tmap(&tdo, a.dctx, kPad, a.head_dim, a.heads, a.S, a.B);
  if (rc) return rc;
  static bool attr_q = false, attr_kv = false;
  rc = set_smem(attention_bwd_dq_kernel<DP, kPad>, bwd_q_smem<DP>(), &attr_q);
  if (rc) return rc;
  rc = set_smem(attention_bwd_dkv_kernel<DP, kPad>, bwd_kv_smem<DP>(), &attr_kv);
  if (rc) return rc;
  const dim3 grid(a.B * a.heads * d.n_tiles);
  cudaError_t le = launch_pdl(attention_bwd_dq_kernel<DP, kPad>, grid, dim3(128), bwd_q_smem<DP>(),
                              stream, tm, tdo, d);
  if (le != cudaSuccess) return static_cast<int>(le);
  le = launch_pdl(attention_bwd_dkv_kernel<DP, kPad>, grid, dim3(128), bwd_kv_smem<DP>(), stream,
                  tm, tdo, d);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}

static_assert(fwd_smem<128>() <= 227 * 1024 && bwd_q_smem<128>() <= 227 * 1024 &&
                  bwd_kv_smem<128>() <= 227 * 1024,
              "DP = 128 tiles exceed the shared memory of one CTA");

}  // namespace

bool attention_supported(int S, int head_dim) {
  return S > 0 && (S % 8) == 0 && (head_dim % 8) == 0 && head_dim >= 8 && head_dim <= 128;
}

int launch_attention_fwd_tiled(const AttnArgs& a, cudaStream_t stream) {
  AttnTDev d;
  int rc = fill_dev(a, &d);
  if (rc) return rc;
  if (a.head_dim == kD) return launch_fwd<64, false>(a, d, stream);
  if (a.head_dim < kD) return launch_fwd<64, true>(a, d, stream);
  return launch_fwd<128, true>(a, d, stream);
}

int launch_attention_bwd_tiled(const AttnArgs& a, cudaStream_t stream) {
  AttnTDev d;
  int rc = fill_dev(a, &d);
  if (rc) return rc;
  if (a.lse == nullptr || a.ctx == nullptr || a.dctx == nullptr || a.dqkv == nullptr) return 931;
  if (a.head_dim == kD) return launch_bwd<64, false>(a, d, stream);
  if (a.head_dim < kD) return launch_bwd<64, true>(a, d, stream);
  return launch_bwd<128, true>(a, d, stream);
}

}  // namespace sky
