// Persistent warp-specialised tcgen05 GEMM for sm_100a (B200).
//
//   out[M,N] = epilogue( sum_k A[m,k] * B[n,k] )      bf16 x bf16 -> fp32 (TMEM) -> bf16 | fp32
//
//   * operands staged by TMA (cp.async.bulk.tensor, SWIZZLE_128B) into a 4..6 deep smem ring,
//   * tcgen05.mma.cta_group::1.kind::f16 (UMMA 128 x BLOCK_N x 16) issued by ONE thread,
//   * two TMEM accumulator buffers (2 x BLOCK_N columns) so the epilogue of tile i overlaps the
//     main loop of tile i+1,
//   * epilogue warps read TMEM with tcgen05.ld, apply bias / erf-GELU / GELU' / dropout /
//     residual add, and store straight to global memory -- which may be the NEXT PIPELINE STAGE's
//     HBM (peer pointer over NVLink); a per-128-row-panel flag is then bumped with
//     red.release.sys so the consumer GPU can start on that panel while we still compute,
//   * symmetric consumer side: the TMA producer can ld.acquire.sys-poll such flags before it
//     loads the A rows of a panel (GEMM -> GEMM boundary), see GemmArgs in api.h.
//
// Both operands may be K-major or MN-major (UMMA descriptor "major" bits), so forward
// (x W^T), dgrad (dy W) and wgrad (dy^T x) all run on this one kernel without transposes.
//
// Reference parity: replaces every nn.Linear / LinearActivation call in
// scaelum/model/bert_layers.py:60-108,227-229,281,311-313,319 and the autograd backward of those.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "api.h"
#include "launch_util.h"
#include "sm100_ptx.cuh"

namespace sky {

namespace {

#ifndef SKY_GEMM_SETMAXNREG
#define SKY_GEMM_SETMAXNREG 0
#endif

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 bytes = one swizzle-128B row
constexpr int UMMA_K = 16;
constexpr int kNumThreads = 384;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 idle, warps4-11 epilogue
constexpr int kEpiWarp0 = 4;
constexpr uint64_t kFlagTimeoutNs = 4000000000ull;  // 4 s

// PAIR: two CTAs (cluster of 2, cta_group::2) compute one 256 x BLOCK_N tile; each stages its own
// 128 rows of A and half of the B tile.
template <int BLOCK_N, bool PAIR>
struct Cfg {
  static constexpr int kBRows = PAIR ? BLOCK_N / 2 : BLOCK_N;  // B rows staged by ONE CTA
  static constexpr int kStages = PAIR ? (BLOCK_N == 256 ? 6 : 8) : (BLOCK_N == 256 ? 4 : 6);
  static constexpr int kABytes = BLOCK_M * BLOCK_K * 2;
  static constexpr int kBBytes = kBRows * BLOCK_K * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = 2 * BLOCK_N;  // 256 or 512 (power of two)
  static constexpr int kBiasBytes = 2 * BLOCK_N * 4;  // double-buffered bias tile
  static constexpr int kOutStageBytes = 8 * 32 * 80;  // per epilogue warp: 32 rows x (64+16) B
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ +
                                    256 /*barriers*/ + kBiasBytes + kOutStageBytes;
};

struct GemmDev {
  int M, N, K;
  void* out;
  void* out2;
  const float* bias;
  const __nv_bfloat16* aux;
  long long ldo, ldo2, ldaux;
  int act;
  int add_aux;
  int accumulate;
  float dropout_p;
  const uint64_t* rng_state;
  uint32_t rng_stream;
  uint32_t* signal_flags;
  const uint32_t* wait_flags;
  const uint32_t* wait_epoch;
  uint32_t wait_mult;
  int* error_flag;
  int debug;
  // stream-K: the flattened (tile, k-block) space is cut into one contiguous range per CTA (pair);
  // tiles shared by several CTAs are reduced through `ws` by whichever CTA arrives last
  int stream_k;
  float* ws;           // partial accumulators: slot (2 * unit + which) * ctas_per_unit + cta_rank
  uint32_t* counters;  // per CTA tile: [2 * t] arrivals, [2 * t + 1] partials written
};

struct Work {
  int tile, kb0, kb1;
};

// Tile scheduler shared by the three warp roles.  Classic mode: tiles unit, unit + U, ... with the
// whole K range.  Stream-K mode: k-blocks [unit * T / U, (unit + 1) * T / U) of T = tiles * nk.
struct Sched {
  int stream, unit, num_units, num_tiles, nk;
  long long total;
  int pos, end, tile;
  __device__ __forceinline__ long long bound(int u) const { return u * total / num_units; }
  __device__ __forceinline__ void init(int stream_k, int unit_, int num_units_, int num_tiles_,
                                       int nk_) {
    stream = stream_k;
    unit = unit_;
    num_units = num_units_;
    num_tiles = num_tiles_;
    nk = nk_;
    total = static_cast<long long>(num_tiles_) * nk_;
    pos = static_cast<int>(bound(unit_));
    end = static_cast<int>(bound(unit_ + 1));
    tile = unit_ - num_units_;
  }
  __device__ __forceinline__ bool next(Work& w) {
    if (!stream) {
      tile += num_units;
      if (tile >= num_tiles) return false;
      w.tile = tile;
      w.kb0 = 0;
      w.kb1 = nk;
      return true;
    }
    if (pos >= end) return false;
    w.tile = pos / nk;
    w.kb0 = pos - w.tile * nk;
    const int len = min(nk - w.kb0, end - pos);
    w.kb1 = w.kb0 + len;
    pos += len;
    return true;
  }
  // unit whose range contains flattened position x
  __device__ __forceinline__ int unit_of(long long x) const {
    int u = static_cast<int>(x * num_units / total);
    while (u + 1 < num_units && bound(u + 1) <= x) ++u;
    while (u > 0 && bound(u) > x) --u;
    return u;
  }
  __device__ __forceinline__ int first_tile(int u) const { return static_cast<int>(bound(u) / nk); }
};

// CL = CTAs per cluster: 1 = independent CTAs, 2 = one cta_group::2 pair, 4 = two pairs that work
// on the same 256 rows and neighbouring N tiles and MULTICAST the A operand to each other (each
// CTA fetches half of its 128 A rows from L2 and TMA delivers them to itself and to the CTA of
// the other pair that needs the same rows).
// SK = stream-K schedule compiled in (a separate instantiation: its bookkeeping costs registers in
// the epilogue, which the classic kernels - the ones every training step runs - must not pay).
template <int BLOCK_N, bool A_MN, bool B_MN, bool OUT_F32, int CL, bool SK>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a,
                    const __grid_constant__ CUtensorMap tmap_b, const GemmDev p) {
  constexpr bool PAIR = CL >= 2;
  constexpr bool MC = CL == 4;
  using C = Cfg<BLOCK_N, PAIR>;
  constexpr int kStages = C::kStages;
  const uint32_t cl_rank = PAIR ? cluster_ctarank() : 0u;  // rank in the cluster
  const uint32_t cta_rank = cl_rank & 1u;                  // rank in the pair
  const uint32_t pair_idx = cl_rank >> 1;                  // which pair of the cluster (MC)
  const uint32_t leader_rank = cl_rank & ~1u;              // cluster rank of this pair's leader
  const bool leader = cta_rank == 0;

  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * C::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * C::kStageBytes);
  uint64_t* full_bar = bars;                       // [kStages]
  uint64_t* empty_bar = bars + kStages;            // [kStages]
  uint64_t* tmem_full_bar = bars + 2 * kStages;    // [2]
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2;  // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);
  float* s_bias = reinterpret_cast<float*>(smem + kStages * C::kStageBytes + 256);

  // warp-uniform by construction AND visibly so to the compiler: the producer / MMA warps run
  // converged with one ELECTED lane issuing, so that TMA / UMMA operands stay in uniform
  // registers.  (A single-lane `if (lane == 0)` role costs an ELECT + 5 R2UR.BROADCAST in front
  // of every UTCHMMA: measured 175 cycles per MMA instead of 64-128, profiles/gemm_schedules.md.)
  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  // tile scheduler: a "unit" is one CTA (128 rows) or one CTA pair (256 rows)
  constexpr int UNIT_M = PAIR ? 2 * BLOCK_M : BLOCK_M;
  const int num_m_units = (p.M + UNIT_M - 1) / UNIT_M;
  const int num_n_blks = (p.N + BLOCK_N - 1) / BLOCK_N;
  // MC: a scheduling unit covers TWO neighbouring N tiles (one per pair); the host only selects
  // this mode when the number of N tiles is even
  const int num_n_units = MC ? num_n_blks / 2 : num_n_blks;
  const int num_tiles = num_m_units * num_n_units;
  const int num_k_blks = (p.K + BLOCK_K - 1) / BLOCK_K;
  const int unit_id = static_cast<int>(blockIdx.x) / CL;
  const int num_units = static_cast<int>(gridDim.x) / CL;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      // MC: a stage is written by two CTAs' multicasts, so BOTH pairs' MMAs must have released it
      mbar_init(&empty_bar[i], MC ? 2 : 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      // one arrive per epilogue warp (of both CTAs in pair mode: the leader's barrier is used)
      mbar_init(&tmem_empty_bar[i], PAIR ? 16 : 8);
    }
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    if constexpr (PAIR) {
      tmem_alloc_pair(tmem_ptr_smem, C::kTmemCols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_ptr_smem, C::kTmemCols);
      tmem_relinquish();
    }
  }
  tcgen05_fence_before();
  __syncwarp();
  if constexpr (PAIR)
    cluster_sync_all();  // the peer's barriers must be initialised before anything signals them
  else
    __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // everything above (barrier init, TMEM alloc, tensormap prefetch) overlapped the previous
  // kernel's tail; from here on we read what it produced
  pdl_wait();
  pdl_launch_dependents();

  // Optional register re-allocation between the warpgroups (setmaxnreg): the producer / MMA /
  // allocator warpgroup keeps 40 registers per thread, the two epilogue warpgroups get 232 (the
  // launch allocation is 384 x 168).  Compile-time experiment, OFF by default: with it ptxas
  // removes the 48-68 byte spill frames of the 256-wide instantiations, but it has not been run
  // on a GPU yet (build with SKY_GEMM_SETMAXNREG=1 in the environment to try it).
#if SKY_GEMM_SETMAXNREG
  if (warp_idx < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
#endif
  if (warp_idx == 0) {
    // ===================================== TMA producer =====================================
    int stage = 0;
    uint32_t phase = 0;
    // pair mode: both CTAs' loads complete on the LEADER's full barrier (cluster address)
    const uint32_t full_addr0 = PAIR ? mapa_shared(smem_u32(&full_bar[0]), leader_rank) : 0u;
    // multicast loads name the barrier by its CTA-relative address with the peer bit cleared:
    // every destination CTA's pair leader receives the bytes that landed in that destination
    const uint32_t full_mc0 = smem_u32(&full_bar[0]) & 0xFEFFFFFFu;
    const uint16_t mc_mask = static_cast<uint16_t>((1u << cl_rank) | (1u << (cl_rank ^ 2u)));
    Sched sched;
    sched.init(SK ? 1 : 0, unit_id, num_units, num_tiles, num_k_blks);
    Work w;
    while (sched.next(w)) {
      const int tile = w.tile;
      const int m_blk = (tile % num_m_units) * (PAIR ? 2 : 1) + static_cast<int>(cta_rank);
      const int n_blk = (tile / num_m_units) * (MC ? 2 : 1) + (MC ? static_cast<int>(pair_idx) : 0);
      const int b_row0 = n_blk * BLOCK_N + static_cast<int>(cta_rank) * C::kBRows;
      if (p.wait_flags != nullptr && m_blk * BLOCK_M < p.M) {
        if (elect_one_sync()) {
          const uint32_t target = (*p.wait_epoch) * p.wait_mult;
          if (!wait_flag_ge(p.wait_flags + m_blk, target, kFlagTimeoutNs)) {
            if (p.error_flag) atomicExch(p.error_flag, 1);
          }
          fence_proxy_async();  // peer generic-proxy writes -> our async-proxy (TMA) reads
        }
        __syncwarp();
      }
      for (int kb = w.kb0; kb < w.kb1; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (!PAIR && p.debug == 3) {  // triage: no loads at all, the MMAs chew on stale smem
          if (elect_one_sync()) mbar_arrive(&full_bar[stage]);
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
          continue;
        }
        if (elect_one_sync()) {
        if (leader) mbar_expect_tx(&full_bar[stage], (PAIR ? 2 : 1) * C::kStageBytes);
        uint8_t* sa = smem_a + stage * C::kABytes;
        uint8_t* sb = smem_b + stage * C::kBBytes;
        auto load = [&](uint8_t* dst, const CUtensorMap* tm, int c0, int c1) {
          if constexpr (PAIR)
            tma_load_2d_pair(dst, tm, full_addr0 + stage * 8, c0, c1);
          else
            tma_load_2d(dst, tm, &full_bar[stage], c0, c1);
        };
        if constexpr (MC) {
          // my half (64 rows) of the A tile, delivered to me and to the CTA of the other pair
          const int h = static_cast<int>(pair_idx);
          if constexpr (!A_MN)
            tma_load_2d_pair_mc(sa + h * (64 * 128), &tmap_a, full_mc0 + stage * 8, kb * BLOCK_K,
                                m_blk * BLOCK_M + h * 64, mc_mask);
          else
            tma_load_2d_pair_mc(sa + h * (BLOCK_K * 128), &tmap_a, full_mc0 + stage * 8,
                                m_blk * BLOCK_M + h * 64, kb * BLOCK_K, mc_mask);
        } else if constexpr (!A_MN) {
          load(sa, &tmap_a, kb * BLOCK_K, m_blk * BLOCK_M);
        } else {
#pragma unroll
          for (int c = 0; c < BLOCK_M / 64; ++c)
            load(sa + c * (BLOCK_K * 128), &tmap_a, m_blk * BLOCK_M + c * 64, kb * BLOCK_K);
        }
        if constexpr (!B_MN) {
          load(sb, &tmap_b, kb * BLOCK_K, b_row0);
        } else {
#pragma unroll
          for (int c = 0; c < C::kBRows / 64; ++c)
            load(sb + c * (BLOCK_K * 128), &tmap_b, b_row0 + c * 64, kb * BLOCK_K);
        }
        }  // elected lane
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp_idx == 1 && leader) {
    // ===================================== MMA issuer ======================================
    constexpr uint32_t idesc = make_idesc_bf16_f32(UNIT_M, BLOCK_N, A_MN, B_MN);
    // K-major  SW128: 8-row atoms 1024B apart (SBO), LBO unused (1); K advance = 32B per UMMA_K
    // MN-major SW128: 64-element MN chunks BLOCK_K*128B apart (LBO), 8-k-row groups 1024B apart
    //                 (SBO); K advance = 16 rows * 128B = 2048B per UMMA_K
    constexpr uint32_t a_lbo = A_MN ? BLOCK_K * 128 : 16;
    constexpr uint32_t b_lbo = B_MN ? BLOCK_K * 128 : 16;
    constexpr uint32_t a_kadv = (A_MN ? UMMA_K * 128 : UMMA_K * 2) >> 4;
    constexpr uint32_t b_kadv = (B_MN ? UMMA_K * 128 : UMMA_K * 2) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    Sched sched;
    sched.init(SK ? 1 : 0, unit_id, num_units, num_tiles, num_k_blks);
    Work w;
    for (; sched.next(w); ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
      for (int kb = w.kb0; kb < w.kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (!PAIR && p.debug == 4) {  // triage: loads only, no MMA
          if (elect_one_sync()) {
            mbar_arrive(&empty_bar[stage]);
            if (kb == w.kb1 - 1) mbar_arrive(&tmem_full_bar[acc]);
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
          continue;
        }
        if (elect_one_sync()) {
        const uint64_t desc_a =
            make_smem_desc_sw128(smem_u32(smem_a + stage * C::kABytes), a_lbo, 1024);
        const uint64_t desc_b =
            make_smem_desc_sw128(smem_u32(smem_b + stage * C::kBBytes), b_lbo, 1024);
#pragma unroll
        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
          if constexpr (PAIR)
            umma_bf16_ss_pair(tmem_d, desc_a + k * a_kadv, desc_b + k * b_kadv, idesc,
                              (kb != w.kb0 || k != 0) ? 1u : 0u);
          else
            umma_bf16_ss(tmem_d, desc_a + k * a_kadv, desc_b + k * b_kadv, idesc,
                         (kb != w.kb0 || k != 0) ? 1u : 0u);
        }
        // smem slot reusable (in both CTAs) once these MMAs retire
        if constexpr (PAIR) {
          const uint16_t pair_mask = static_cast<uint16_t>(3u << leader_rank);
          umma_commit_pair(&empty_bar[stage], MC ? static_cast<uint16_t>(0xF) : pair_mask);
          if (kb == w.kb1 - 1) umma_commit_pair(&tmem_full_bar[acc], pair_mask);
        } else {
          umma_commit(&empty_bar[stage]);
          if (kb == w.kb1 - 1) umma_commit(&tmem_full_bar[acc]);
        }
        }  // elected lane
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
#if SKY_GEMM_SETMAXNREG
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    {
#else
  } else if (warp_idx >= kEpiWarp0) {
#endif
    // ====================================== epilogue =======================================
    // 8 warps: warp e handles TMEM lane quadrant (e & 3) and column half (e >> 2) of the tile.
    // Latency hiding (profiles/gemm_epilogue_v1.md: the first version stalled ~80% on
    // long-scoreboard waits for bias/aux global loads with one warp per scheduler):
    //   * bias for the tile is staged once in shared memory (double buffered per accumulator),
    //   * aux (residual / pre-activation) chunks are prefetched one chunk ahead, the first one
    //     before the accumulator is even ready,
    //   * TMEM loads are double buffered: chunk c+1 is in flight while chunk c is processed,
    //   * fp32 gradient accumulation uses red.global.add.v4.f32 (no read-modify-write).
    const int e = warp_idx - kEpiWarp0;
    const int q = e & 3;  // == warp_idx % 4: the TMEM lanes this warp may access
    const int half = e >> 2;
    constexpr int HALF_N = BLOCK_N / 2;
    constexpr int NCH = HALF_N / 32;
    const int epi_tid = threadIdx.x - kEpiWarp0 * 32;  // 0..255
    uint8_t* s_stage = smem + kStages * C::kStageBytes + 256 + C::kBiasBytes + e * (32 * 80);
    const int row_in_tile = q * 32 + lane;
    const bool has_dropout = p.dropout_p > 0.f;
    const bool has_aux = p.aux != nullptr;
    uint64_t seed = 0;
    uint32_t thr16 = 0;
    float drop_scale = 1.f;
    if (has_dropout) {
      seed = dropout_seed(p.rng_state, p.rng_stream);
      thr16 = static_cast<uint32_t>(p.dropout_p * 65536.f);
      drop_scale = 1.f / (1.f - p.dropout_p);
    }
    int it = 0;
    const uint32_t tmem_empty_addr0 =
        PAIR ? mapa_shared(smem_u32(&tmem_empty_bar[0]), leader_rank)
             : smem_u32(&tmem_empty_bar[0]);
    Sched sched;
    sched.init(SK ? 1 : 0, unit_id, num_units, num_tiles, num_k_blks);
    Work w;
    uint32_t* s_ticket = tmem_ptr_smem + 1;
    constexpr int kCtasPerUnit = CL;
    constexpr int kTileElems = BLOCK_M * BLOCK_N;
    for (; sched.next(w); ++it) {
      const int tile = w.tile;
      const int m_blk = (tile % num_m_units) * (PAIR ? 2 : 1) + static_cast<int>(cta_rank);
      const int n_blk = (tile / num_m_units) * (MC ? 2 : 1) + (MC ? static_cast<int>(pair_idx) : 0);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const long long row = static_cast<long long>(m_blk) * BLOCK_M + row_in_tile;
      const bool row_ok = row < p.M;
      const int colbase = n_blk * BLOCK_N + half * HALF_N;
      // ---- stage bias, prefetch first aux chunk (both overlap the MMA main loop) ----
      float* sb = s_bias + acc * BLOCK_N;
      if (epi_tid < BLOCK_N) {
        const int gc = n_blk * BLOCK_N + epi_tid;
        sb[epi_tid] = (p.bias != nullptr && gc < p.N) ? __ldg(p.bias + gc) : 0.f;
      }
      uint4 auxa[4], auxb[4];
      const __nv_bfloat16* aux_row = has_aux ? p.aux + row * p.ldaux + colbase : nullptr;
      auto load_aux = [&](uint4 (&dst)[4], int c) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int col = colbase + c * 32 + t * 8;
          dst[t] = (has_aux && row_ok && col < p.N)
                       ? *reinterpret_cast<const uint4*>(aux_row + c * 32 + t * 8)
                       : make_uint4(0, 0, 0, 0);
        }
      };
      if (has_aux) load_aux(auxa, 0);
      asm volatile("bar.sync 1, 256;" ::: "memory");  // bias of this tile visible to all 8 warps

      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr =
          tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N + half * HALF_N;

      // ---- stream-K: is this CTA the one that finishes the tile? ----
      // Every contributor takes a ticket once its share of the K range sits in TMEM.  All but the
      // last arrival park their raw fp32 accumulators in the workspace and bump `done`; the last
      // arrival waits for those writes (the writers are already past their main loop, so the
      // wait is short and cannot deadlock), adds them and runs the real epilogue.
      bool finisher = true;
      int n_contrib = 1, u_first = 0;
      float* ws_mine = nullptr;
      const bool partial = SK && !(w.kb0 == 0 && w.kb1 == num_k_blks) && !p.accumulate;
      const int ctile = n_blk * (num_m_units * (PAIR ? 2 : 1)) + m_blk;
      if (partial) {
        u_first = sched.unit_of(static_cast<long long>(tile) * num_k_blks);
        const int u_last = sched.unit_of(static_cast<long long>(tile + 1) * num_k_blks - 1);
        n_contrib = u_last - u_first + 1;
        if (epi_tid == 0) *s_ticket = atomicAdd(p.counters + 2 * ctile, 1u);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        finisher = (*s_ticket == static_cast<uint32_t>(n_contrib - 1));
        const int which = (tile == sched.first_tile(unit_id)) ? 0 : 1;
        ws_mine = p.ws + static_cast<size_t>((2 * unit_id + which) * kCtasPerUnit + cl_rank) *
                             kTileElems;
        if (finisher) {
          if (epi_tid == 0) {
            const uint64_t t0 = globaltimer_ns();
            while (ld_acquire_sys(p.counters + 2 * ctile + 1) <
                   static_cast<uint32_t>(n_contrib - 1)) {
              if (globaltimer_ns() - t0 > kFlagTimeoutNs) {
                if (p.error_flag) atomicExch(p.error_flag, 2);
                break;
              }
            }
            p.counters[2 * ctile] = 0;  // leave the counters clean for the next launch
            p.counters[2 * ctile + 1] = 0;
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
      }
      // workspace layout of one 128 x BLOCK_N tile: [column / 4][row][4] floats, so that the 32
      // lanes (= 32 rows) of a warp touch 512 contiguous bytes per float4 access
      auto ws_ptr = [&](float* base, int c) {
        return reinterpret_cast<float4*>(base) + ((half * HALF_N + c * 32) >> 2) * BLOCK_M +
               row_in_tile;
      };

      // bf16 stores go through a per-warp smem transpose: a lane owns one accumulator ROW, so
      // storing straight from registers makes every STG.128 touch 32 different rows (32 partial
      // sectors per request).  Staged, a warp store covers 8 rows x 64 contiguous bytes.
      // Row stride 80 B keeps both the row-wise writes and the 4-lanes-per-row reads (nearly)
      // bank-conflict free.
      const long long warp_row0 = static_cast<long long>(m_blk) * BLOCK_M + q * 32;
      auto store_bf16_chunk = [&](const float (&f)[32], __nv_bfloat16* gout, long long ld,
                                  int col0) {
        uint8_t* mine = s_stage + lane * 80;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 pk;
          pk.x = pack_bf16x2(f[j], f[j + 1]);
          pk.y = pack_bf16x2(f[j + 2], f[j + 3]);
          pk.z = pack_bf16x2(f[j + 4], f[j + 5]);
          pk.w = pack_bf16x2(f[j + 6], f[j + 7]);
          *reinterpret_cast<uint4*>(mine + j * 2) = pk;
        }
        __syncwarp();
        const int piece = lane & 3;
        if (col0 + piece * 8 < p.N) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = i * 8 + (lane >> 2);
            if (warp_row0 + r < p.M) {
              const uint4 val = *reinterpret_cast<const uint4*>(s_stage + r * 80 + piece * 16);
              *reinterpret_cast<uint4*>(gout + (warp_row0 + r) * ld + col0 + piece * 8) = val;
            }
          }
        }
        __syncwarp();
      };

      auto process = [&](uint32_t (&v)[32], uint4 (&ax)[4], int c) {
        const int col0 = colbase + c * 32;
        if (col0 >= p.N || p.debug == 1 || p.debug >= 3) return;  // warp-uniform
        if (partial) {
          if (!finisher) {
            float4* wp = ws_ptr(ws_mine, c);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              wp[j * BLOCK_M] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                            __uint_as_float(v[4 * j + 2]),
                                            __uint_as_float(v[4 * j + 3]));
            return;
          }
          for (int u = u_first; u < u_first + n_contrib; ++u) {
            if (u == unit_id) continue;
            const int which_u = (tile == sched.first_tile(u)) ? 0 : 1;
            const float4* rp = ws_ptr(
                p.ws + static_cast<size_t>((2 * u + which_u) * kCtasPerUnit + cl_rank) * kTileElems,
                c);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 x = __ldcg(rp + j * BLOCK_M);
              v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + x.x);
              v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + x.y);
              v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + x.z);
              v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + x.w);
            }
          }
        }
        float f[32];
        const float4* sb4 = reinterpret_cast<const float4*>(sb + half * HALF_N + c * 32);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 bb = sb4[j >> 2];  // smem broadcast
          f[j] = __uint_as_float(v[j]) + bb.x;
          f[j + 1] = __uint_as_float(v[j + 1]) + bb.y;
          f[j + 2] = __uint_as_float(v[j + 2]) + bb.z;
          f[j + 3] = __uint_as_float(v[j + 3]) + bb.w;
        }
        if (p.act == ACT_GELU) {
          if (p.out2 != nullptr && p.debug != 2)
            store_bf16_chunk(f, reinterpret_cast<__nv_bfloat16*>(p.out2), p.ldo2, col0);
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = gelu_fast(f[j]);
        } else if (p.act == ACT_TANH) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = tanh_fast(f[j]);
        }
        if (has_dropout) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const uint64_t idx4 = (static_cast<uint64_t>(row) * p.N + col0 + j) >> 2;
            const uint32_t m = dropout_keep4(seed, idx4, thr16);
            f[j] = (m & 1u) ? f[j] * drop_scale : 0.f;
            f[j + 1] = (m & 2u) ? f[j + 1] * drop_scale : 0.f;
            f[j + 2] = (m & 4u) ? f[j + 2] * drop_scale : 0.f;
            f[j + 3] = (m & 8u) ? f[j + 3] * drop_scale : 0.f;
          }
        }
        if (has_aux) {
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint32_t aw[4] = {ax[t].x, ax[t].y, ax[t].z, ax[t].w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 x = unpack_bf16x2(aw[u]);
              const int j = t * 8 + u * 2;
              if (p.act == ACT_DGELU_MUL_AUX) {
                f[j] *= dgelu_fast(x.x);
                f[j + 1] *= dgelu_fast(x.y);
              } else if (p.add_aux) {
                f[j] += x.x;
                f[j + 1] += x.y;
              }
            }
          }
        }
        if (p.debug != 2) {
          if constexpr (OUT_F32) {
            if (row_ok) {
              float* o = reinterpret_cast<float*>(p.out) + row * p.ldo + col0;
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                if (col0 + j < p.N) {
                  if (p.accumulate)
                    red_add_v4_f32(o + j, f[j], f[j + 1], f[j + 2], f[j + 3]);
                  else
                    *reinterpret_cast<float4*>(o + j) =
                        make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                }
              }
            }
          } else {
            store_bf16_chunk(f, reinterpret_cast<__nv_bfloat16*>(p.out), p.ldo, col0);
          }
        }
      };

      uint32_t va[32], vb[32];
      tmem_ld_32x32b_x32(taddr, va);
#pragma unroll 1
      for (int c = 0; c < NCH; c += 2) {
        tmem_ld_wait();                                // chunk c landed in va
        tmem_ld_32x32b_x32(taddr + (c + 1) * 32, vb);  // chunk c+1 in flight
        if (has_aux) load_aux(auxb, c + 1);
        process(va, auxa, c);
        tmem_ld_wait();  // chunk c+1 landed in vb
        if (c + 2 < NCH) {
          tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
          if (has_aux) load_aux(auxa, c + 2);
        }
        process(vb, auxb, c + 1);
      }
      // release the TMEM buffer back to the MMA warp
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR)
          mbar_arrive_cluster(tmem_empty_addr0 + acc * 8);
        else
          mbar_arrive(&tmem_empty_bar[acc]);
      }
      if (partial && !finisher) {
        // publish the parked partial: all stores -> fence -> barrier -> one counter bump
        __threadfence();
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (epi_tid == 0) atomicAdd(p.counters + 2 * ctile + 1, 1u);
      }
      if (finisher && p.signal_flags != nullptr && m_blk * BLOCK_M < p.M) {
        // publish this tile: all 256 epilogue threads' stores -> barrier -> one release.sys
        __threadfence_system();
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (epi_tid == 0) red_release_sys_add(p.signal_flags + m_blk, 1u);
      }
    }
  }

#if SKY_GEMM_SETMAXNREG
  }
#endif

  tcgen05_fence_before();
  __syncwarp();
  if constexpr (PAIR)
    cluster_sync_all();  // neither CTA may leave while the other still signals / reads it
  else
    __syncthreads();
  if (warp_idx == 2) {
    tcgen05_fence_after();
    if constexpr (PAIR)
      tmem_dealloc_pair(tmem_base, C::kTmemCols);
    else
      tmem_dealloc(tmem_base, C::kTmemCols);
  }
}


// ------------------------------------------------------------------------------------------
// GEMM + bias + dropout + residual + LayerNorm in ONE kernel (SURVEY K4 / K6):
//
//     y = LayerNorm( dropout(A W^T + bias) + residual ) * gamma + beta        z = the pre-LN sum
//
// A LayerNorm row spans all N columns, a CTA's accumulator only BLOCK_N of them, so the N / BLOCK_N
// CTAs that own the column tiles of one 128-row panel form a THREAD-BLOCK CLUSTER (2..8 CTAs) and
// exchange per-row partial sums through distributed shared memory:
//
//   pass 1  TMEM -> registers: + bias, dropout, + residual; store z (bf16, saved for backward);
//           accumulate row sum / sum of squares; write the fp32 values BACK into the accumulator's
//           own TMEM columns (tcgen05.st) - 128 x BLOCK_N fp32 do not fit in registers
//   DSMEM   every row-owner thread stores its (sum, sumsq) into ALL CTAs of the cluster
//           (st.shared::cluster) and arrives on their mbarriers (release.cluster)
//   pass 2  TMEM -> registers again: normalise with the cluster-wide statistics, gamma / beta,
//           store y - straight into the NEXT PIPELINE STAGE's HBM when y is a peer pointer, then
//           one red.release.sys per CTA on the panel flag.
//
// This is the forward stage boundary of the north star: the last GEMM of stage i stores its
// output tiles into stage i+1's HBM from inside the tcgen05 kernel; no separate LayerNorm launch.
// Reference ops replaced: scaelum/model/bert_layers.py:285-289 (BertSelfOutput) and :323-327
// (BertOutput); hop replaced: scaelum/builder/module_wrapper.py:148-175.
// ------------------------------------------------------------------------------------------
struct GemmLnDev {
  int M, N, K;
  void* y;
  void* z;
  long long ldy, ldz, ldaux;
  const float* bias;
  const __nv_bfloat16* aux;
  const float* gamma;
  const float* beta;
  float* mean;
  float* rstd;
  float eps;
  float dropout_p;
  const uint64_t* rng_state;
  uint32_t rng_stream;
  uint32_t* signal_flags;
  const uint32_t* wait_flags;
  const uint32_t* wait_epoch;
  uint32_t wait_mult;
  int* error_flag;
};

constexpr int kLnMaxCluster = 8;

template <int BLOCK_N>
struct LnCfg {
  using C = Cfg<BLOCK_N, false>;
  static constexpr int kStages = C::kStages;
  static constexpr int kVecBytes = 3 * BLOCK_N * 4;                 // bias, gamma, beta
  static constexpr int kStatsBytes = kLnMaxCluster * BLOCK_M * 8;   // float2 per (cta, row)
  static constexpr int kOffBars = kStages * C::kStageBytes;
  static constexpr int kOffVec = kOffBars + 256;
  static constexpr int kOffOut = kOffVec + kVecBytes;
  static constexpr int kOffStats = kOffOut + C::kOutStageBytes;
  static constexpr int kSmemBytes = kOffStats + kStatsBytes + 1024 /*align slack*/;
};

template <int BLOCK_N>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_ln_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a,
                       const __grid_constant__ CUtensorMap tmap_b, const GemmLnDev p) {
  using L = LnCfg<BLOCK_N>;
  using C = typename L::C;
  constexpr int kStages = L::kStages;
  const uint32_t cln = cluster_nctarank();     // CTAs per cluster == column tiles per row panel
  const uint32_t n_blk = cluster_ctarank();    // this CTA's column tile
  const int m_blk = static_cast<int>(blockIdx.x / cln);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * C::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kOffBars);
  uint64_t* full_bar = bars;               // [kStages]
  uint64_t* empty_bar = bars + kStages;    // [kStages]
  uint64_t* tmem_full_bar = bars + 2 * kStages;
  uint64_t* stats_bar = bars + 2 * kStages + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 2);
  float* s_bias = reinterpret_cast<float*>(smem + L::kOffVec);
  float* s_gamma = s_bias + BLOCK_N;
  float* s_beta = s_gamma + BLOCK_N;
  float2* s_stats = reinterpret_cast<float2*>(smem + L::kOffStats);   // [cln][128]

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int num_k_blks = (p.K + BLOCK_K - 1) / BLOCK_K;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(stats_bar, cln * BLOCK_M);   // one arrival per row-owner thread of every CTA
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc(tmem_ptr_smem, BLOCK_N);
    tmem_relinquish();
  }
  tcgen05_fence_before();
  __syncwarp();
  cluster_sync_all();   // peers' stats barriers exist before anybody arrives on them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();
  pdl_launch_dependents();

  if (warp_idx == 0) {
    // ===================================== TMA producer =====================================
    int stage = 0;
    uint32_t phase = 0;
    if (p.wait_flags != nullptr) {
      if (elect_one_sync()) {
        const uint32_t target = (*p.wait_epoch) * p.wait_mult;
        if (!wait_flag_ge(p.wait_flags + m_blk, target, kFlagTimeoutNs)) {
          if (p.error_flag) atomicExch(p.error_flag, 1);
        }
        fence_proxy_async();
      }
      __syncwarp();
    }
    for (int kb = 0; kb < num_k_blks; ++kb) {
      mbar_wait(&empty_bar[stage], phase ^ 1);
      if (elect_one_sync()) {
        mbar_expect_tx(&full_bar[stage], C::kStageBytes);
        tma_load_2d(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], kb * BLOCK_K,
                    m_blk * BLOCK_M);
        tma_load_2d(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BLOCK_K,
                    static_cast<int>(n_blk) * BLOCK_N);
      }
      __syncwarp();
      if (++stage == kStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp_idx == 1) {
    // ===================================== MMA issuer ======================================
    constexpr uint32_t idesc = make_idesc_bf16_f32(BLOCK_M, BLOCK_N, false, false);
    constexpr uint32_t kadv = (UMMA_K * 2) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = 0; kb < num_k_blks; ++kb) {
      mbar_wait(&full_bar[stage], phase);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint64_t desc_a = make_smem_desc_sw128(smem_u32(smem_a + stage * C::kABytes), 16, 1024);
        const uint64_t desc_b = make_smem_desc_sw128(smem_u32(smem_b + stage * C::kBBytes), 16, 1024);
#pragma unroll
        for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
          umma_bf16_ss(tmem_base, desc_a + k * kadv, desc_b + k * kadv, idesc,
                       (kb != 0 || k != 0) ? 1u : 0u);
        umma_commit(&empty_bar[stage]);
        if (kb == num_k_blks - 1) umma_commit(tmem_full_bar);
      }
      __syncwarp();
      if (++stage == kStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp_idx >= kEpiWarp0) {
    // ====================================== epilogue =======================================
    const int e = warp_idx - kEpiWarp0;
    const int q = e & 3;
    const int half = e >> 2;
    constexpr int HALF_N = BLOCK_N / 2;
    constexpr int NCH = HALF_N / 32;
    const int epi_tid = threadIdx.x - kEpiWarp0 * 32;
    uint8_t* s_out = smem + L::kOffOut;
    uint8_t* s_stage = s_out + e * (32 * 80);
    const int row_in_tile = q * 32 + lane;
    const long long row = static_cast<long long>(m_blk) * BLOCK_M + row_in_tile;
    const bool row_ok = row < p.M;
    const int colbase = static_cast<int>(n_blk) * BLOCK_N + half * HALF_N;
    const bool has_dropout = p.dropout_p > 0.f;
    const bool has_aux = p.aux != nullptr;
    uint64_t seed = 0;
    uint32_t thr16 = 0;
    float drop_scale = 1.f;
    if (has_dropout) {
      seed = dropout_seed(p.rng_state, p.rng_stream);
      thr16 = static_cast<uint32_t>(p.dropout_p * 65536.f);
      drop_scale = 1.f / (1.f - p.dropout_p);
    }
    for (int i = epi_tid; i < BLOCK_N; i += 256) {
      const int gc = static_cast<int>(n_blk) * BLOCK_N + i;
      s_bias[i] = p.bias != nullptr ? __ldg(p.bias + gc) : 0.f;
      s_gamma[i] = __ldg(p.gamma + gc);
      s_beta[i] = __ldg(p.beta + gc);
    }
    uint4 auxa[4], auxb[4];
    const __nv_bfloat16* aux_row = has_aux ? p.aux + row * p.ldaux + colbase : nullptr;
    auto load_aux = [&](uint4 (&dst)[4], int c) {
#pragma unroll
      for (int t = 0; t < 4; ++t)
        dst[t] = (has_aux && row_ok)
                     ? *reinterpret_cast<const uint4*>(aux_row + c * 32 + t * 8)
                     : make_uint4(0, 0, 0, 0);
    };
    if (has_aux) load_aux(auxa, 0);
    asm volatile("bar.sync 1, 256;" ::: "memory");

    const long long warp_row0 = static_cast<long long>(m_blk) * BLOCK_M + q * 32;
    auto store_bf16_chunk = [&](const float (&f)[32], __nv_bfloat16* gout, long long ld, int col0) {
      uint8_t* mine = s_stage + lane * 80;
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 pk;
        pk.x = pack_bf16x2(f[j], f[j + 1]);
        pk.y = pack_bf16x2(f[j + 2], f[j + 3]);
        pk.z = pack_bf16x2(f[j + 4], f[j + 5]);
        pk.w = pack_bf16x2(f[j + 6], f[j + 7]);
        *reinterpret_cast<uint4*>(mine + j * 2) = pk;
      }
      __syncwarp();
      const int piece = lane & 3;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = i * 8 + (lane >> 2);
        if (warp_row0 + r < p.M) {
          const uint4 val = *reinterpret_cast<const uint4*>(s_stage + r * 80 + piece * 16);
          *reinterpret_cast<uint4*>(gout + (warp_row0 + r) * ld + col0 + piece * 8) = val;
        }
      }
      __syncwarp();
    };

    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + half * HALF_N;

    // ---------------- pass 1: z = dropout(acc + bias) + residual; row statistics ----------------
    float s1 = 0.f, s2 = 0.f;
    auto pass1 = [&](uint32_t (&v)[32], uint4 (&ax)[4], int c) {
      const int col0 = colbase + c * 32;
      float f[32];
      const float4* sb4 = reinterpret_cast<const float4*>(s_bias + half * HALF_N + c * 32);
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 bb = sb4[j >> 2];
        f[j] = __uint_as_float(v[j]) + bb.x;
        f[j + 1] = __uint_as_float(v[j + 1]) + bb.y;
        f[j + 2] = __uint_as_float(v[j + 2]) + bb.z;
        f[j + 3] = __uint_as_float(v[j + 3]) + bb.w;
      }
      if (has_dropout) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const uint64_t idx4 = (static_cast<uint64_t>(row) * p.N + col0 + j) >> 2;
          const uint32_t m = dropout_keep4(seed, idx4, thr16);
          f[j] = (m & 1u) ? f[j] * drop_scale : 0.f;
          f[j + 1] = (m & 2u) ? f[j + 1] * drop_scale : 0.f;
          f[j + 2] = (m & 4u) ? f[j + 2] * drop_scale : 0.f;
          f[j + 3] = (m & 8u) ? f[j + 3] * drop_scale : 0.f;
        }
      }
      if (has_aux) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t aw[4] = {ax[t].x, ax[t].y, ax[t].z, ax[t].w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float2 x = unpack_bf16x2(aw[u]);
            f[t * 8 + u * 2] += x.x;
            f[t * 8 + u * 2 + 1] += x.y;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        s1 += f[j];
        s2 = fmaf(f[j], f[j], s2);
        v[j] = __float_as_uint(f[j]);
      }
      tmem_st_32x32b_x32(taddr + c * 32, v);   // park the fp32 sum in the accumulator's columns
      if (p.z != nullptr)
        store_bf16_chunk(f, reinterpret_cast<__nv_bfloat16*>(p.z), p.ldz, col0);
    };
    {
      uint32_t va[32], vb[32];
      tmem_ld_32x32b_x32(taddr, va);
#pragma unroll 1
      for (int c = 0; c < NCH; c += 2) {
        tmem_ld_wait();
        tmem_ld_32x32b_x32(taddr + (c + 1) * 32, vb);
        if (has_aux) load_aux(auxb, c + 1);
        pass1(va, auxa, c);
        tmem_ld_wait();
        if (c + 2 < NCH) {
          tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
          if (has_aux) load_aux(auxa, c + 2);
        }
        pass1(vb, auxb, c + 1);
      }
      tmem_st_wait();
    }
    // ---------------- cluster-wide row statistics through distributed shared memory ----------------
    // the two column halves of a row live in warps e and e + 4: combine them through the (now
    // idle) output staging area, then the half-0 thread of each row publishes to every CTA
    float2* s_half = reinterpret_cast<float2*>(s_out);
    asm volatile("bar.sync 1, 256;" ::: "memory");   // every warp is done with its staging slice
    if (half == 1) s_half[row_in_tile] = make_float2(s1, s2);
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (half == 0) {
      const float2 o = s_half[row_in_tile];
      s1 += o.x;
      s2 += o.y;
      const uint32_t slot = smem_u32(&s_stats[n_blk * BLOCK_M + row_in_tile]);
      const uint32_t bar = smem_u32(stats_bar);
      for (uint32_t r = 0; r < cln; ++r) {
        st_cluster_v2_f32(mapa_shared(slot, r), s1, s2);
        mbar_arrive_cluster(mapa_shared(bar, r));
      }
    }
    mbar_wait_cluster(stats_bar, 0);
    float t1 = 0.f, t2 = 0.f;
    for (uint32_t r = 0; r < cln; ++r) {
      const float2 o = s_stats[r * BLOCK_M + row_in_tile];
      t1 += o.x;
      t2 += o.y;
    }
    const float inv_n = 1.f / static_cast<float>(p.N);
    const float mean = t1 * inv_n;
    const float var = fmaxf(fmaf(-mean, mean, t2 * inv_n), 0.f);
    const float rstd = rsqrtf(var + p.eps);
    if (n_blk == 0 && half == 0 && row_ok) {
      p.mean[row] = mean;
      p.rstd[row] = rstd;
    }
    // ---------------- pass 2: normalise, gamma / beta, store y (possibly into a peer GPU) ----------------
    auto pass2 = [&](const uint32_t (&v)[32], int c) {
      const int col0 = colbase + c * 32;
      float f[32];
      const float4* g4 = reinterpret_cast<const float4*>(s_gamma + half * HALF_N + c * 32);
      const float4* b4 = reinterpret_cast<const float4*>(s_beta + half * HALF_N + c * 32);
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 g = g4[j >> 2], b = b4[j >> 2];
        f[j] = fmaf((__uint_as_float(v[j]) - mean) * rstd, g.x, b.x);
        f[j + 1] = fmaf((__uint_as_float(v[j + 1]) - mean) * rstd, g.y, b.y);
        f[j + 2] = fmaf((__uint_as_float(v[j + 2]) - mean) * rstd, g.z, b.z);
        f[j + 3] = fmaf((__uint_as_float(v[j + 3]) - mean) * rstd, g.w, b.w);
      }
      store_bf16_chunk(f, reinterpret_cast<__nv_bfloat16*>(p.y), p.ldy, col0);
    };
    {
      uint32_t va[32], vb[32];
      tmem_ld_32x32b_x32(taddr, va);
#pragma unroll 1
      for (int c = 0; c < NCH; c += 2) {
        tmem_ld_wait();
        tmem_ld_32x32b_x32(taddr + (c + 1) * 32, vb);
        pass2(va, c);
        tmem_ld_wait();
        if (c + 2 < NCH) tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
        pass2(vb, c + 1);
      }
    }
    if (p.signal_flags != nullptr) {
      // publish this CTA's 128 x BLOCK_N tile of the panel: stores -> fence -> barrier -> one
      // release.sys; the consumer waits for epoch x (N / BLOCK_N) signals per panel
      __threadfence_system();
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (epi_tid == 0) red_release_sys_add(p.signal_flags + m_blk, 1u);
    }
  }

  tcgen05_fence_before();
  __syncwarp();
  cluster_sync_all();   // nobody leaves while a peer may still write its statistics into us
  if (warp_idx == 2) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, BLOCK_N);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e =
        cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  });
  return fn;
}

}  // namespace

// 2D bf16 tensor map: inner (contiguous) extent `inner`, `outer` rows of stride ld elements.
int make_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t outer,
                      uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return 901;
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstride[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 1000 + static_cast<int>(r);
}

// 3D bf16 tensor map (inner, middle, outer) for [outer][middle][inner] data: the attention kernels
// view the [B * S, C] activations as (C, S, B) so that a 128-row box never crosses a sequence.
int make_tmap_bf16_3d(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t middle,
                      uint64_t outer, uint64_t ld_middle_elems, uint64_t ld_outer_elems,
                      uint32_t box_inner, uint32_t box_middle) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return 901;
  cuuint64_t gdim[3] = {inner, middle, outer};
  cuuint64_t gstride[2] = {ld_middle_elems * 2, ld_outer_elems * 2};
  cuuint32_t box[3] = {box_inner, box_middle, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gdim, gstride,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 1000 + static_cast<int>(r);
}

// 4D bf16 tensor map, dims[0] contiguous, ld_elems[i] = stride of dims[i + 1]; box
// (box_inner, 1, box_third, 1).  The attention kernels view [B * S, sections * D] activations as
// (D, sections, S, B): a box wider than D then reads zeros past the end of a head's columns.
int make_tmap_bf16_4d(CUtensorMap* tm, const void* ptr, const uint64_t (&dims)[4],
                      const uint64_t (&ld_elems)[3], uint32_t box_inner, uint32_t box_third) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return 901;
  cuuint64_t gdim[4] = {dims[0], dims[1], dims[2], dims[3]};
  cuuint64_t gstride[3] = {ld_elems[0] * 2, ld_elems[1] * 2, ld_elems[2] * 2};
  cuuint32_t box[4] = {box_inner, 1, box_third, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), gdim, gstride,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 1000 + static_cast<int>(r);
}

int gemm_pick_block_n(int M, int N) {
  // 256-wide tiles halve B re-reads and give the best tensor-pipe duty cycle; fall back to 128
  // when that would leave most SMs idle or N is small.
  const long long tiles256 = static_cast<long long>((M + 127) / 128) * ((N + 255) / 256);
  if (N % 256 != 0 && N <= 128) return 128;
  if (tiles256 < 96) return 128;
  return 256;
}

bool gemm_pick_quad(int M, int N, int K) {
  // Two cta_group::2 pairs per cluster with the A operand multicast between them.  Measured
  // (profiles/gemm_schedules.md): wins 20-25 % on the few-tile, deep-K shapes that pick 128-wide
  // tiles (dgrads / FFN2 at <= 2048 tokens, attn_out wgrad), loses on everything else.
  static int env = -2;
  if (env == -2) {
    const char* e = std::getenv("SKY_GEMM_QUAD");
    env = e ? std::atoi(e) : -1;
  }
  if (env == 0) return false;
  if (env > 0) return true;
  return M >= 256 && K >= 2048 && gemm_pick_block_n(M, N) == 128 && ((N + 127) / 128) % 2 == 0;
}

bool gemm_pick_pair(int M, int N, int K) {
  (void)N;
  (void)K;
  static int env = -2;
  if (env == -2) {
    const char* e = std::getenv("SKY_GEMM_PAIR");
    env = e ? std::atoi(e) : -1;
  }
  if (env >= 0) return env != 0 && M > 128;
  return false;  // measured: the TPC already merges the two SMs' identical B requests
}

int gemm_tiles_per_panel(int N, int block_n) { return (N + block_n - 1) / block_n; }

namespace {
static int g_num_sms = 0;

// ---- stream-K workspace: one per (device, stream), because GEMMs on different streams overlap ----
constexpr size_t kWsSlotBytes = static_cast<size_t>(BLOCK_M) * 256 * 4;  // one 128 x 256 fp32 tile
constexpr int kWsMaxCtas = 160;                                          // >= SMs of the device
constexpr int kWsMaxCtaTiles = 8192;
struct StreamKWs {
  float* ws = nullptr;
  uint32_t* counters = nullptr;
};
std::mutex g_ws_mutex;
std::map<std::pair<int, cudaStream_t>, StreamKWs> g_ws;

// nullptr when the workspace does not exist yet and cannot be created (stream is capturing)
const StreamKWs* get_ws(cudaStream_t stream) {
  int dev_id = 0;
  cudaGetDevice(&dev_id);
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  auto key = std::make_pair(dev_id, stream);
  auto it = g_ws.find(key);
  if (it != g_ws.end()) return &it->second;
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) {
    cudaGetLastError();
    return nullptr;
  }
  StreamKWs w;
  if (cudaMalloc(&w.ws, 2 * kWsMaxCtas * kWsSlotBytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (cudaMalloc(&w.counters, 2 * kWsMaxCtaTiles * sizeof(uint32_t)) != cudaSuccess) {
    cudaGetLastError();
    cudaFree(w.ws);
    return nullptr;
  }
  cudaMemset(w.counters, 0, 2 * kWsMaxCtaTiles * sizeof(uint32_t));
  g_ws[key] = w;
  return &g_ws[key];
}

// Stream-K pays when the classic schedule leaves SMs idle (few tiles) or ends on a ragged wave:
// compare ceil(tiles / U) * nk against tiles * nk / U k-blocks per CTA (+ a fix-up allowance).
bool want_stream_k(long long tiles, int nk, int units, bool accumulate) {
  static int env = -2;
  if (env == -2) {
    const char* e = std::getenv("SKY_GEMM_STREAMK");
    env = e ? std::atoi(e) : -1;
  }
  if (env == 0) return false;
  if (tiles <= 0 || nk < 8) return false;
  const long long classic = (tiles + units - 1) / units * nk;
  const long long streamed = (tiles * nk + units - 1) / units + 6;
  if (streamed < 4) return false;
  if (env == 1) return tiles % units != 0;
  // Measured (profiles/gemm_schedules.md): the fix-up of split tiles (park + re-read 128 KB per
  // CTA, finisher wait) costs more than the idle SMs it recovers on every BERT shape, and with
  // >= units/2 tiles the chip-wide L2 -> SM rate is the limit anyway.  It pays for fp32 `+=`
  // outputs (weight gradients: partials are red.add'ed, no fix-up) with few tiles and a deep K.
  // ... in isolation (attn_out wgrad 27 -> 17 us).  Inside the training step those weight
  // gradients run on the side stream NEXT TO the dgrad chain, where a 148-CTA stream-K grid takes
  // SMs away from the critical path: 12.62 ms/step with it, 12.50 ms without => opt-in only.
  (void)accumulate;
  return false;
}

template <int BLOCK_N, bool A_MN, bool B_MN, bool OUT_F32, int CL>
int launch_inst(const GemmArgs& a, const GemmDev& dev, cudaStream_t stream) {
  constexpr bool PAIR = CL >= 2;
  constexpr bool MC = CL == 4;
  using C = Cfg<BLOCK_N, PAIR>;
  CUtensorMap tma, tmb;
  int rc;
  if (!A_MN)
    rc = make_tmap_bf16_2d(&tma, a.A, a.K, a.M, a.lda, BLOCK_K, MC ? 64 : BLOCK_M);
  else
    rc = make_tmap_bf16_2d(&tma, a.A, a.M, a.K, a.lda, 64, BLOCK_K);
  if (rc) return rc;
  if (!B_MN)
    rc = make_tmap_bf16_2d(&tmb, a.B, a.K, a.N, a.ldb, BLOCK_K, C::kBRows);
  else
    rc = make_tmap_bf16_2d(&tmb, a.B, a.N, a.K, a.ldb, 64, BLOCK_K);
  if (rc) return rc;

  GemmDev devp = dev;
  {
    if (g_num_sms == 0) {
      int dev_id = 0;
      cudaGetDevice(&dev_id);
      cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev_id);
    }
    constexpr int UM = PAIR ? 2 * BLOCK_M : BLOCK_M;
    const long long m_units = (a.M + UM - 1) / UM;
    const long long n_blks = (a.N + BLOCK_N - 1) / BLOCK_N;
    const long long tiles = m_units * (MC ? n_blks / 2 : n_blks);
    const int nk = (a.K + BLOCK_K - 1) / BLOCK_K;
    int units = g_num_sms / CL;
    if (a.max_ctas > 0 && units > a.max_ctas / CL) units = a.max_ctas / CL;
    if (units < 1) units = 1;
    bool sk = a.stream_k < 0 ? want_stream_k(tiles, nk, units, a.accumulate) : (a.stream_k != 0);
    // every CTA must own at least 4 k-blocks, the CTA tiles must fit the counter array, a bias
    // must not be added once per partial, and the grid must fit the workspace
    if (tiles * nk < 4LL * units) sk = false;
    if (m_units * (PAIR ? 2 : 1) * n_blks > kWsMaxCtaTiles || g_num_sms > kWsMaxCtas) sk = false;
    if (a.accumulate && a.bias != nullptr) sk = false;
    devp.stream_k = 0;
    devp.ws = nullptr;
    devp.counters = nullptr;
    if (sk) {
      if (a.accumulate) {
        devp.stream_k = 1;  // partial sums go straight to the fp32 output with red.add
      } else if (const StreamKWs* w = get_ws(stream)) {
        devp.stream_k = 1;
        devp.ws = w->ws;
        devp.counters = w->counters;
      }
    }
  }
  // stream-K instantiations exist for independent CTAs only (pairs / clusters did not profit)
  if (CL != 1) devp.stream_k = 0;
  void (*kern)(CUtensorMap, CUtensorMap, GemmDev) =
      gemm_tcgen05_kernel<BLOCK_N, A_MN, B_MN, OUT_F32, CL, false>;
  if constexpr (CL == 1) {
    if (devp.stream_k) kern = gemm_tcgen05_kernel<BLOCK_N, A_MN, B_MN, OUT_F32, CL, true>;
  }
  static bool attr_set[2] = {false, false};
  if (!attr_set[devp.stream_k ? 1 : 0]) {
    cudaError_t e =
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set[devp.stream_k ? 1 : 0] = true;
  }
  if (g_num_sms == 0) {
    int dev_id = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev_id);
  }
  constexpr int UNIT_M = PAIR ? 2 * BLOCK_M : BLOCK_M;
  const int num_tiles =
      ((a.M + UNIT_M - 1) / UNIT_M) * (((a.N + BLOCK_N - 1) / BLOCK_N) / (MC ? 2 : 1));
  const int max_units = g_num_sms / CL;
  int grid = (num_tiles < max_units && !devp.stream_k) ? num_tiles : max_units;
  if (a.max_ctas > 0 && grid > a.max_ctas / CL) grid = a.max_ctas / CL;
  if (grid < 1) grid = 1;
  grid *= CL;
  cudaError_t le = launch_pdl_cluster(kern, dim3(grid), dim3(kNumThreads), C::kSmemBytes, stream,
                              CL, tma, tmb, devp);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}

template <int BLOCK_N, int PAIR>
int dispatch_major(const GemmArgs& a, const GemmDev& dev, cudaStream_t stream) {
  if (!a.a_mn && !a.b_mn)
    return a.out_f32 ? launch_inst<BLOCK_N, false, false, true, PAIR>(a, dev, stream)
                     : launch_inst<BLOCK_N, false, false, false, PAIR>(a, dev, stream);
  if (!a.a_mn && a.b_mn)
    return a.out_f32 ? launch_inst<BLOCK_N, false, true, true, PAIR>(a, dev, stream)
                     : launch_inst<BLOCK_N, false, true, false, PAIR>(a, dev, stream);
  if (a.a_mn && a.b_mn)
    return a.out_f32 ? launch_inst<BLOCK_N, true, true, true, PAIR>(a, dev, stream)
                     : launch_inst<BLOCK_N, true, true, false, PAIR>(a, dev, stream);
  return a.out_f32 ? launch_inst<BLOCK_N, true, false, true, PAIR>(a, dev, stream)
                   : launch_inst<BLOCK_N, true, false, false, PAIR>(a, dev, stream);
}
}  // namespace


// ---- GEMM + LayerNorm epilogue: tile width, cluster size ----
int gemm_ln_block_n(int M, int N, bool force) {
  // 0 = do not run the fused kernel for this shape.  Measured on B200 (profiles/gemm_ln.md):
  // 256-wide tiles in 4-CTA clusters beat GEMM + standalone LayerNorm by 12 % once the launch
  // fills the GPU (>= 96 CTAs, i.e. >= 3072 tokens at N = 1024); with fewer tokens the two-kernel
  // path's 128-wide GEMM tiles use twice as many SMs and win, and 128-wide tiles in 8-CTA clusters
  // lose outright (at most one such cluster fits a GPC next to another: 29 vs 15 us at 2048
  // tokens).  `force` (tests, SKY_FUSE_LN=force) accepts every shape the kernel can run.
  if (M <= 0 || N <= 0 || (N % 128) != 0) return 0;
  const long long panels = (M + 127) / 128;
  const bool ok256 = (N % 256) == 0 && N / 256 <= kLnMaxCluster;
  const bool ok128 = N / 128 <= kLnMaxCluster;
  if (ok256 && panels * (N / 256) >= 96) return 256;
  if (!force) return 0;
  if (ok256) return 256;
  return ok128 ? 128 : 0;
}
int gemm_ln_tiles_per_panel(int M, int N, bool force) {
  const int bn = gemm_ln_block_n(M, N, force);
  return bn ? N / bn : 0;
}

namespace {
template <int BLOCK_N>
int launch_ln_inst(const GemmArgs& a, const GemmLnDev& dev, cudaStream_t stream) {
  using L = LnCfg<BLOCK_N>;
  using C = typename L::C;
  CUtensorMap tma, tmb;
  int rc = make_tmap_bf16_2d(&tma, a.A, a.K, a.M, a.lda, BLOCK_K, BLOCK_M);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmb, a.B, a.K, a.N, a.ldb, BLOCK_K, C::kBRows);
  if (rc) return rc;
  void (*kern)(CUtensorMap, CUtensorMap, GemmLnDev) = gemm_ln_tcgen05_kernel<BLOCK_N>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         L::kSmemBytes);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_set = true;
  }
  const int cln = a.N / BLOCK_N;
  const int panels = (a.M + BLOCK_M - 1) / BLOCK_M;
  cudaError_t le = launch_pdl_cluster(kern, dim3(panels * cln), dim3(kNumThreads), L::kSmemBytes,
                                      stream, cln, tma, tmb, dev);
  if (le != cudaSuccess) return static_cast<int>(le);
  return static_cast<int>(cudaGetLastError());
}
}  // namespace

int launch_gemm_ln(const GemmArgs& a, cudaStream_t stream) {
  if (a.M <= 0 || a.N <= 0 || a.K <= 0) return 0;
  if (a.a_mn || a.b_mn || a.out_f32 || a.accumulate || a.act != ACT_NONE) return 908;
  if ((a.K % 8) != 0 || (a.lda % 8) != 0 || (a.ldb % 8) != 0) return 902;
  if (a.ln_gamma == nullptr || a.ln_beta == nullptr || a.ln_mean == nullptr ||
      a.ln_rstd == nullptr || a.out == nullptr)
    return 909;
  if (a.dropout_p > 0.f && a.rng_state == nullptr) return 903;
  if (a.aux != nullptr && !a.add_aux) return 908;
  const int bn = a.block_n ? a.block_n : gemm_ln_block_n(a.M, a.N, true);
  if (bn == 0 || (a.N % bn) != 0 || a.N / bn > kLnMaxCluster) return 907;
  GemmLnDev d;
  d.M = a.M;
  d.N = a.N;
  d.K = a.K;
  d.y = a.out;
  d.ldy = a.ldo;
  d.z = a.out2;
  d.ldz = a.ldo2;
  d.bias = a.bias;
  d.aux = reinterpret_cast<const __nv_bfloat16*>(a.aux);
  d.ldaux = a.ldaux;
  d.gamma = a.ln_gamma;
  d.beta = a.ln_beta;
  d.mean = a.ln_mean;
  d.rstd = a.ln_rstd;
  d.eps = a.ln_eps;
  d.dropout_p = a.dropout_p;
  d.rng_state = a.rng_state;
  d.rng_stream = a.rng_stream;
  d.signal_flags = a.signal_flags;
  d.wait_flags = a.wait_flags;
  d.wait_epoch = a.wait_epoch;
  d.wait_mult = a.wait_mult;
  d.error_flag = a.error_flag;
  if (bn == 256) return launch_ln_inst<256>(a, d, stream);
  if (bn == 128) return launch_ln_inst<128>(a, d, stream);
  return 905;
}

int launch_gemm(const GemmArgs& a, cudaStream_t stream) {
  if (a.M <= 0 || a.N <= 0 || a.K <= 0) return 0;
  if (a.ln_gamma != nullptr) return launch_gemm_ln(a, stream);
  if ((a.N % 8) != 0 || (a.K % 8) != 0 || (a.lda % 8) != 0 || (a.ldb % 8) != 0) return 902;
  if (a.a_mn && (a.M % 8) != 0) return 902;
  if (a.dropout_p > 0.f && a.rng_state == nullptr) return 903;
  if (a.accumulate && !a.out_f32) return 904;
  GemmDev d;
  d.M = a.M;
  d.N = a.N;
  d.K = a.K;
  d.out = a.out;
  d.out2 = a.out2;
  d.bias = a.bias;
  d.aux = reinterpret_cast<const __nv_bfloat16*>(a.aux);
  d.ldo = a.ldo;
  d.ldo2 = a.ldo2;
  d.ldaux = a.ldaux;
  d.act = a.act;
  d.add_aux = a.add_aux ? 1 : 0;
  d.accumulate = a.accumulate ? 1 : 0;
  d.dropout_p = a.dropout_p;
  d.rng_state = a.rng_state;
  d.rng_stream = a.rng_stream;
  d.signal_flags = a.signal_flags;
  d.wait_flags = a.wait_flags;
  d.wait_epoch = a.wait_epoch;
  d.wait_mult = a.wait_mult;
  d.error_flag = a.error_flag;
  d.debug = a.debug;
  d.stream_k = 0;
  d.ws = nullptr;
  d.counters = nullptr;
  const int bn = a.block_n ? a.block_n : gemm_pick_block_n(a.M, a.N);
  const bool auto_quad = a.pair < 0 && a.block_n == 0 && gemm_pick_quad(a.M, a.N, a.K);
  const bool pair = a.pair < 0 ? (auto_quad || gemm_pick_pair(a.M, a.N, a.K)) : (a.pair != 0);
  if (pair) {
    // two pairs + A multicast needs an even number of N tiles
    const bool quad = (a.pair == 2 || auto_quad) &&
                      (((a.N + bn - 1) / bn) % 2 == 0);
    if (quad) {
      if (bn == 256) return dispatch_major<256, 4>(a, d, stream);
      if (bn == 128) return dispatch_major<128, 4>(a, d, stream);
      return 905;
    }
    if (bn == 256) return dispatch_major<256, 2>(a, d, stream);
    if (bn == 128) return dispatch_major<128, 2>(a, d, stream);
    return 905;
  }
  if (bn == 256) return dispatch_major<256, 1>(a, d, stream);
  if (bn == 128) return dispatch_major<128, 1>(a, d, stream);
  return 905;
}

}  // namespace sky
