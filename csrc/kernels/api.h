// C++ launch API of the sm_100a kernel library (no torch dependency: compiled by nvcc alone,
// bound to Python in csrc/bindings.cpp).  All launchers are asynchronous on `stream`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sky {

// ---------------------------------------------------------------------------------------------
// GEMM  out[M,N] = epilogue( sum_k A[m,k] * B[n,k] )   bf16 operands, fp32 accumulation in TMEM
// ---------------------------------------------------------------------------------------------
enum GemmAct : int { ACT_NONE = 0, ACT_GELU = 1, ACT_DGELU_MUL_AUX = 2, ACT_TANH = 3 };

struct GemmArgs {
  const void* A = nullptr;  // bf16
  const void* B = nullptr;  // bf16
  int M = 0, N = 0, K = 0;
  // a_mn == false: A stored row-major [M, K] (K contiguous), lda = row stride in elements
  // a_mn == true : A stored row-major [K, M] (M contiguous), lda = row stride in elements
  int lda = 0, ldb = 0;
  bool a_mn = false, b_mn = false;

  void* out = nullptr;  // bf16 (default) or fp32 when out_f32; may be a peer-GPU pointer
  int ldo = 0;
  bool out_f32 = false;
  bool accumulate = false;  // out += result (fp32 outputs only)
  void* out2 = nullptr;     // optional bf16 copy of the pre-activation (bias added)
  int ldo2 = 0;

  const float* bias = nullptr;  // [N] fp32
  const void* aux = nullptr;    // bf16 [M,N]: residual (add_aux) or pre-activation (DGELU_MUL_AUX)
  int ldaux = 0;
  int act = ACT_NONE;
  bool add_aux = false;

  float dropout_p = 0.f;                // applied after bias/activation, before add_aux
  const uint64_t* rng_state = nullptr;  // device: {seed, step}; required when dropout_p > 0
  uint32_t rng_stream = 0;              // per-call-site stream id

  // Stage-boundary fusion.  signal_flags[m_blk] (possibly in peer memory) is incremented with
  // release.sys semantics once per finished output tile.  wait_flags[m_blk] (local memory) is
  // polled with acquire.sys by the TMA producer before it loads A rows of that 128-row panel; the
  // expected value is (*wait_epoch) * wait_mult.
  uint32_t* signal_flags = nullptr;
  const uint32_t* wait_flags = nullptr;
  const uint32_t* wait_epoch = nullptr;
  uint32_t wait_mult = 0;
  int* error_flag = nullptr;  // set to non-zero on flag-wait timeout
  // LayerNorm epilogue (ln_gamma != nullptr): out = LN(dropout(A B^T + bias) + aux) * gamma + beta,
  // out2 = the pre-LN sum (bf16, saved for backward), ln_mean / ln_rstd = row statistics.  The
  // N / BLOCK_N CTAs of a 128-row panel form a thread-block cluster (row statistics through
  // DSMEM); `out` may be peer memory, signal_flags[panel] then receives N / BLOCK_N signals.
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
  float* ln_mean = nullptr;
  float* ln_rstd = nullptr;
  float ln_eps = 1e-12f;
  int block_n = 0;            // 0 = auto (128 or 256)
  int stream_k = -1;          // stream-K schedule: -1 auto, 0 off, 1 on
  int pair = -1;              // -1 auto, 0 single CTAs, 1 cta_group::2 pairs, 2 = 4-CTA clusters: two pairs + A multicast
  int debug = 0;              // perf triage: 1 = epilogue discards the tile, 2 = epilogue math but no stores
  int max_ctas = 0;           // 0 = all SMs
};

// Returns 0 on success, a cudaError_t / CUresult-like code otherwise.
int launch_gemm(const GemmArgs& args, cudaStream_t stream);
int launch_gemm_ln(const GemmArgs& args, cudaStream_t stream);
// tile width the fused LN epilogue would use (0 = use GEMM + standalone LayerNorm instead; with
// `force` only when the kernel cannot run the shape at all) / signals per 128-row panel
int gemm_ln_block_n(int M, int N, bool force = false);
int gemm_ln_tiles_per_panel(int M, int N, bool force = false);
int gemm_tiles_per_panel(int N, int block_n);  // number of signals per 128-row panel
int gemm_pick_block_n(int M, int N);
bool gemm_pick_pair(int M, int N, int K);
bool gemm_pick_quad(int M, int N, int K);

// ---------------------------------------------------------------------------------------------
// LayerNorm (rows of H), bf16 in/out, fp32 statistics
// ---------------------------------------------------------------------------------------------
struct LayerNormFwdArgs {
  const void* z = nullptr;  // bf16 [M,H]
  void* y = nullptr;        // bf16 [M,H]
  float* mean = nullptr;    // [M]
  float* rstd = nullptr;    // [M]
  const float* gamma = nullptr;
  const float* beta = nullptr;
  int M = 0, H = 0;
  float eps = 1e-12f;
  // optional: wait for 128-row panels written by a peer
  const uint32_t* wait_flags = nullptr;
  const uint32_t* wait_epoch = nullptr;
  uint32_t wait_mult = 0;
  int* error_flag = nullptr;
  // optional: y is (peer) boundary memory; every CTA (8 rows) bumps signal_flags[row/128] once
  // with release.sys, i.e. a 128-row panel is complete at 16 signals (kLnSignalsPerPanel)
  uint32_t* signal_flags = nullptr;
};
constexpr int kLnSignalsPerPanel = 16;
int launch_layernorm_fwd(const LayerNormFwdArgs& a, cudaStream_t stream);

struct LayerNormBwdArgs {
  const void* dy = nullptr;  // bf16 [M,H]
  const void* z = nullptr;   // bf16 [M,H] pre-LN input saved by forward
  const float* mean = nullptr;
  const float* rstd = nullptr;
  const float* gamma = nullptr;
  void* dz = nullptr;         // bf16 [M,H]
  void* dz_dropped = nullptr; // optional bf16 [M,H]: dz * keep/(1-p) with the GEMM-epilogue mask
  float* dgamma = nullptr;    // fp32 [H], accumulated (+=)
  float* dbeta = nullptr;     // fp32 [H], accumulated (+=)
  int M = 0, H = 0;
  float dropout_p = 0.f;
  const uint64_t* rng_state = nullptr;
  uint32_t rng_stream = 0;
  const uint32_t* wait_flags = nullptr;
  const uint32_t* wait_epoch = nullptr;
  uint32_t wait_mult = 0;
  int* error_flag = nullptr;
};
int launch_layernorm_bwd(const LayerNormBwdArgs& a, cudaStream_t stream);
int launch_ln_param_grad(const void* dy, const void* z, const float* mean, const float* rstd,
                         float* dgamma, float* dbeta, int M, int H, const void* x2, float* out2,
                         cudaStream_t stream);

// y[i] = g[i] * gelu'(h[i])  (bf16, n % 8 == 0): only used when a stage cut separates FFN1 | FFN2
int launch_dgelu_mul(const void* g, const void* h, void* y, long long n, cudaStream_t stream);

// column sums: out[n] += sum_m x[m,n]   (bias gradients)
int launch_colsum(const void* x_bf16, int M, int N, int ldx, float* out, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Attention, tcgen05: any S % 8 == 0 and head_dim % 8 == 0 with 8 <= head_dim <= 128 (S = 128 with
// head_dim = 64: single-tile kernels; everything else tiled); other shapes return 930
// ---------------------------------------------------------------------------------------------
struct AttnArgs {
  const void* qkv = nullptr;   // bf16 [B*S, 3*H]  (Q | K | V), head h at columns h*head_dim
  const float* mask = nullptr; // fp32 additive [B, S] or null
  void* ctx = nullptr;         // bf16 [B*S, H] (fwd: output, bwd: saved forward output)
  float* lse = nullptr;        // fp32 [B*heads, S] log2-domain log-sum-exp (fwd: out, bwd: in)
  const void* dctx = nullptr;  // bwd: bf16 [B*S, H]
  void* dqkv = nullptr;        // bwd: bf16 [B*S, 3*H]
  int B = 0, S = 0, heads = 0, head_dim = 0;
  float scale = 0.125f;
  float dropout_p = 0.f;
  const uint64_t* rng_state = nullptr;
  uint32_t rng_stream = 0;
};
int launch_attention_fwd(const AttnArgs& a, cudaStream_t stream);
int launch_attention_bwd(const AttnArgs& a, cudaStream_t stream);
// every supported shape (flash-style tiling over 128-key blocks; backward = dQ kernel + dK/dV kernel)
int launch_attention_fwd_tiled(const AttnArgs& a, cudaStream_t stream);
int launch_attention_bwd_tiled(const AttnArgs& a, cudaStream_t stream);
bool attention_supported(int S, int head_dim);

// ---------------------------------------------------------------------------------------------
// Embeddings: word + position + token-type gather, LayerNorm, dropout; and its backward
// ---------------------------------------------------------------------------------------------
struct EmbedArgs {
  const int64_t* input_ids = nullptr;   // [B*S]
  const int64_t* token_type = nullptr;  // [B*S]
  const int64_t* attn_mask = nullptr;   // [B*S] (0/1) or null
  const float* word = nullptr;          // [V,H] fp32 master weights
  const float* pos = nullptr;           // [P,H]
  const float* type = nullptr;          // [T,H]
  const float* gamma = nullptr;
  const float* beta = nullptr;
  void* out = nullptr;        // bf16 [B*S,H]
  float* ext_mask = nullptr;  // fp32 [B*S] = (1-mask)*-10000
  float* xhat = nullptr;      // optional fp32? (unused) kept null
  float* mean = nullptr;      // [B*S]
  float* rstd = nullptr;      // [B*S]
  int B = 0, S = 0, H = 0;
  float eps = 1e-12f;
  float dropout_p = 0.f;
  const uint64_t* rng_state = nullptr;
  uint32_t rng_stream = 0;
};
int launch_embed_fwd(const EmbedArgs& a, cudaStream_t stream);

struct EmbedBwdArgs {
  const void* dout = nullptr;  // bf16 [B*S,H]
  const int64_t* input_ids = nullptr;
  const int64_t* token_type = nullptr;
  const float* word = nullptr;
  const float* pos = nullptr;
  const float* type = nullptr;
  const float* gamma = nullptr;
  const float* mean = nullptr;
  const float* rstd = nullptr;
  float* dword = nullptr;  // fp32 [V,H] (+=, atomics)
  float* dpos = nullptr;
  float* dtype_ = nullptr;
  float* dgamma = nullptr;
  float* dbeta = nullptr;
  int B = 0, S = 0, H = 0;
  int type_rows = 2;  // rows of the token-type table (accumulated in shared memory when <= 4)
  float dropout_p = 0.f;
  const uint64_t* rng_state = nullptr;
  uint32_t rng_stream = 0;
  const uint32_t* wait_flags = nullptr;
  const uint32_t* wait_epoch = nullptr;
  uint32_t wait_mult = 0;
  int* error_flag = nullptr;
};
int launch_embed_bwd(const EmbedBwdArgs& a, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Small dense layers (pooler / classifier) + softmax cross-entropy, CUDA-core (latency bound)
// ---------------------------------------------------------------------------------------------
// y[m,n] = act( sum_k x[m*ldx + k] * w[n,k] + b[n] ); x bf16 or fp32, w/b fp32, y fp32
int launch_small_linear_fwd(const void* x, bool x_bf16, int ldx, const float* w, const float* b,
                            float* y, int M, int N, int K, int act_tanh, float dropout_p,
                            const uint64_t* rng_state, uint32_t rng_stream, cudaStream_t stream);
// dx[m,k] = sum_n dy'[m,n] w[n,k];  dw[n,k] += sum_m dy'[m,n] x[m,k];  db[n] += sum_m dy'[m,n]
// where dy' = dy * (1 - y^2) if act_tanh.  Input dropout mask is re-applied to x and dx.
int launch_small_linear_bwd(const void* x, bool x_bf16, int ldx, const float* w, const float* y,
                            const float* dy, void* dx, bool dx_bf16, int lddx, float* dw, float* db,
                            int M, int N, int K, int act_tanh, float dropout_p,
                            const uint64_t* rng_state, uint32_t rng_stream, cudaStream_t stream);
// loss = mean_m CE(logits[m,:], labels[m]);  dlogits = (softmax - onehot) / M * grad_scale
int launch_softmax_ce(const float* logits, const int64_t* labels, float* loss, float* dlogits,
                      int M, int C, float grad_scale, float* loss_acc, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Optimizer / parameter maintenance
// ---------------------------------------------------------------------------------------------
// Multi-tensor fused SGD: p -= lr * (g + wd * p) (optional momentum buffer), then refresh the
// bf16 compute copy and zero the gradient.  `n_tensors` descriptors in device memory.
struct SgdTensor {
  float* p;
  float* g;
  float* mom;         // may be null
  void* p_bf16;       // may be null
  long long numel;
  int skip_zero;      // the first gradient write of the next step OVERWRITES g: do not zero it
  int pad_;
  float* mom2;        // Adam second moment (null for SGD)
};
int launch_sgd_multi(const SgdTensor* d_tensors, int n_tensors, long long max_numel, float lr,
                     float momentum, float weight_decay, float grad_scale, bool zero_grad,
                     cudaStream_t stream);
// Multi-tensor fused Adam / AdamW (torch.optim.Adam(W) semantics, amsgrad=False): moments in
// `mom` / `mom2`, the step count lives in DEVICE memory (`step`, advanced by the caller with
// launch_advance_counter before this launch) so that the whole update is CUDA-graph capturable.
int launch_adam_multi(const SgdTensor* d_tensors, int n_tensors, long long max_numel, float lr,
                      float beta1, float beta2, float eps, float weight_decay, bool decoupled,
                      const uint64_t* step, float grad_scale, bool zero_grad, cudaStream_t stream);
int launch_cast_f32_to_bf16(const float* src, void* dst, long long n, cudaStream_t stream);
int launch_cast_bf16_to_f32(const void* src, float* dst, long long n, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Runtime helpers
// ---------------------------------------------------------------------------------------------
int launch_advance_counter(uint64_t* counter, uint64_t inc, cudaStream_t stream);   // rng step
int launch_advance_epoch(uint32_t* counter, uint32_t inc, cudaStream_t stream);     // flag epochs
int launch_signal_flags(uint32_t* flags, int n, uint32_t inc, cudaStream_t stream); // release.sys
int launch_wait_flags(const uint32_t* flags, int n, const uint32_t* epoch, uint32_t mult,
                      int* error_flag, cudaStream_t stream);
// Device-side throttle used by the stimulator / `slowdown`: spins for `ns` nanoseconds, or for
// factor * (elapsed since *t_start_ns) when factor > 0 (simulated slow device).
int launch_spin_ns(uint64_t ns, cudaStream_t stream);
int launch_record_time(uint64_t* slot, cudaStream_t stream);
int launch_spin_factor(const uint64_t* t_start_slot, float factor, cudaStream_t stream);
// Peer copy with flags (unfused boundary over NVLink): copies n bytes (16B multiple) to dst
// (peer pointer) and bumps `n_flags` counters with release.sys.
int launch_peer_copy_signal(const void* src, void* dst, long long nbytes, uint32_t* flags,
                            int n_flags, uint32_t inc, cudaStream_t stream);

}  // namespace sky
