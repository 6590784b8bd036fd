#include "device_bench.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <stdexcept>
#include <string>
#include <vector>

#include "../kernels/api.h"

namespace sky {

namespace {
void ck(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}
void ckrc(int rc, const char* what) {
  if (rc != 0) throw std::runtime_error(std::string(what) + " rc=" + std::to_string(rc));
}
}  // namespace

// The proxy workload IS a transformer block of the model being allocated: the same kernel chain
// BertSpanFn launches for forward + backward (ops/functions.py) - QKV GEMM, tcgen05 attention,
// attention-output GEMM (+ LayerNorm: fused epilogue or standalone kernel, whichever the training
// step would pick for this token count), FFN1 + GELU, FFN2 (+ LayerNorm); then LayerNorm backward
// x 2, the four dgrad and four wgrad GEMMs, attention backward and the bias / LayerNorm parameter
// reductions.  `mode` 0 = that full chain (default), 1 = the four forward GEMMs only (round-1
// proxy, kept for comparison).  The reference times 10 x Conv2d forward with host timers and no
// warm-up (scaelum/dynamics/estimator.py:15-34, experiment/config.py:133-149); a device whose
// attention / memory-bound kernels are slow relative to its GEMMs is mis-ranked by such a proxy.
std::pair<double, double> device_benchmark(int tokens, int hidden, int intermediate, int iterations,
                                           int warmup, double slowdown, int mode, int seq,
                                           int heads, int head_dim) {
  const size_t M = tokens, H = hidden, I = intermediate;
  const bool full = mode == 0 && heads > 0 && hidden == heads * head_dim &&
                    attention_supported(seq, head_dim) && tokens % seq == 0;
  std::vector<void*> allocs;
  auto dmalloc = [&](size_t bytes, int fill) {
    void* p = nullptr;
    ck(cudaMalloc(&p, bytes), "malloc");
    // small non-zero operands (value pattern irrelevant for timing, avoid denormals / NaN)
    ck(cudaMemset(p, fill, bytes), "memset");
    allocs.push_back(p);
    return p;
  };
  auto bf = [&](size_t n, int fill = 0x3c) { return static_cast<__nv_bfloat16*>(dmalloc(n * 2, fill)); };
  auto f32 = [&](size_t n) { return static_cast<float*>(dmalloc(n * 4, 0)); };
  __nv_bfloat16 *x = bf(M * H), *wqkv = bf(3 * H * H), *qkv = bf(M * 3 * H), *wo = bf(H * H),
                *h1 = bf(M * H), *w1 = bf(I * H), *inter = bf(M * I), *w2 = bf(H * I),
                *out = bf(M * H);
  float* bias = f32(3 * H > I ? 3 * H : I);
  uint64_t* tslot = static_cast<uint64_t*>(dmalloc(sizeof(uint64_t), 0));
  // forward + backward extras
  __nv_bfloat16 *ctx = nullptr, *z1 = nullptr, *z2 = nullptr, *pre = nullptr, *dy = nullptr,
                *dz = nullptr, *dh1 = nullptr, *da = nullptr, *dctx = nullptr, *dqkv = nullptr,
                *dx = nullptr;
  float *lse = nullptr, *mean = nullptr, *rstd = nullptr, *gamma = nullptr, *beta = nullptr,
        *gw_qkv = nullptr, *gw_o = nullptr, *gw_1 = nullptr, *gw_2 = nullptr, *gvec = nullptr;
  if (full) {
    ctx = bf(M * H); z1 = bf(M * H); z2 = bf(M * H); pre = bf(M * I); dy = bf(M * H, 0x30);
    dz = bf(M * H); dh1 = bf(M * I); da = bf(M * H); dctx = bf(M * H); dqkv = bf(M * 3 * H);
    dx = bf(M * H);
    lse = f32(static_cast<size_t>(tokens / seq) * heads * seq);
    mean = f32(M); rstd = f32(M); gamma = f32(H); beta = f32(H);
    gw_qkv = f32(3 * H * H); gw_o = f32(H * H); gw_1 = f32(I * H); gw_2 = f32(H * I);
    gvec = f32(3 * H > I ? 3 * H : I);
    std::vector<float> ones(H, 1.f);
    ck(cudaMemcpy(gamma, ones.data(), H * 4, cudaMemcpyHostToDevice), "memcpy");
  }

  cudaStream_t s;
  ck(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "stream");
  cudaEvent_t e0, e1;
  ck(cudaEventCreate(&e0), "event");
  ck(cudaEventCreate(&e1), "event");
  const bool fuse_ln = full && gemm_ln_block_n(tokens, hidden) != 0;

  auto gemm = [&](const void* A, int lda, bool a_mn, const void* B, int ldb, bool b_mn, int m,
                  int n, int k, void* o, int ldo, bool f32out, const char* what) {
    GemmArgs g;
    g.A = A; g.lda = lda; g.a_mn = a_mn; g.B = B; g.ldb = ldb; g.b_mn = b_mn;
    g.M = m; g.N = n; g.K = k; g.out = o; g.ldo = ldo; g.out_f32 = f32out;
    g.accumulate = f32out;
    ckrc(launch_gemm(g, s), what);
  };
  auto dense_ln = [&](const void* A, int lda, const void* W, int k, const void* res, void* z,
                      const char* what) {
    GemmArgs g;
    g.A = A; g.lda = lda; g.B = W; g.ldb = k; g.M = tokens; g.N = hidden; g.K = k;
    g.bias = bias; g.aux = res; g.ldaux = hidden; g.add_aux = true;
    if (fuse_ln) {
      g.out = out; g.ldo = hidden; g.out2 = z; g.ldo2 = hidden;
      g.ln_gamma = gamma; g.ln_beta = beta; g.ln_mean = mean; g.ln_rstd = rstd;
      ckrc(launch_gemm(g, s), what);
    } else {
      g.out = z; g.ldo = hidden;
      ckrc(launch_gemm(g, s), what);
      LayerNormFwdArgs l;
      l.z = z; l.y = out; l.mean = mean; l.rstd = rstd; l.gamma = gamma; l.beta = beta;
      l.M = tokens; l.H = hidden;
      ckrc(launch_layernorm_fwd(l, s), "layernorm_fwd");
    }
  };
  auto ln_bwd = [&](const void* z) {
    LayerNormBwdArgs l;
    l.dy = dy; l.z = z; l.mean = mean; l.rstd = rstd; l.gamma = gamma; l.dz = dz;
    l.M = tokens; l.H = hidden;
    ckrc(launch_layernorm_bwd(l, s), "layernorm_bwd");
    ckrc(launch_ln_param_grad(dy, z, mean, rstd, gvec, gvec, tokens, hidden, dz, gvec, s),
         "ln_param_grad");
  };

  auto block = [&]() {
    GemmArgs g;
    g.M = tokens;
    g.bias = bias;
    // QKV
    g.A = x; g.lda = hidden; g.B = wqkv; g.ldb = hidden; g.N = 3 * hidden; g.K = hidden;
    g.out = qkv; g.ldo = 3 * hidden; g.act = ACT_NONE;
    ckrc(launch_gemm(g, s), "gemm qkv");
    if (!full) {
      // attention output projection (A = first H columns of qkv as a stand-in for ctx)
      g.A = qkv; g.lda = 3 * hidden; g.B = wo; g.ldb = hidden; g.N = hidden; g.K = hidden;
      g.out = h1; g.ldo = hidden;
      ckrc(launch_gemm(g, s), "gemm attn-out");
    } else {
      AttnArgs a;
      a.qkv = qkv; a.ctx = ctx; a.lse = lse; a.B = tokens / seq; a.S = seq; a.heads = heads;
      a.head_dim = head_dim;
      ckrc(launch_attention_fwd(a, s), "attention_fwd");
      dense_ln(ctx, hidden, wo, hidden, x, z1, "gemm attn-out (+LN)");
      ck(cudaMemcpyAsync(h1, out, M * H * 2, cudaMemcpyDeviceToDevice, s), "copy");
    }
    // FFN1 + GELU
    g.A = h1; g.lda = hidden; g.B = w1; g.ldb = hidden; g.N = intermediate; g.K = hidden;
    g.out = inter; g.ldo = intermediate; g.act = ACT_GELU;
    g.out2 = full ? pre : nullptr; g.ldo2 = intermediate;
    ckrc(launch_gemm(g, s), "gemm ffn1");
    g.out2 = nullptr;
    // FFN2
    if (!full) {
      g.A = inter; g.lda = intermediate; g.B = w2; g.ldb = intermediate; g.N = hidden;
      g.K = intermediate; g.out = out; g.ldo = hidden; g.act = ACT_NONE;
      ckrc(launch_gemm(g, s), "gemm ffn2");
      return;
    }
    dense_ln(inter, intermediate, w2, intermediate, h1, z2, "gemm ffn2 (+LN)");
    // ------------------------------- backward -------------------------------
    ln_bwd(z2);
    gemm(dz, hidden, true, inter, intermediate, true, hidden, intermediate, tokens, gw_2,
         intermediate, true, "wgrad ffn2");
    {  // FFN2 dgrad x GELU'
      GemmArgs d;
      d.A = dz; d.lda = hidden; d.B = w2; d.ldb = intermediate; d.b_mn = true; d.M = tokens;
      d.N = intermediate; d.K = hidden; d.out = dh1; d.ldo = intermediate; d.aux = pre;
      d.ldaux = intermediate; d.act = ACT_DGELU_MUL_AUX;
      ckrc(launch_gemm(d, s), "dgrad ffn2");
    }
    gemm(dh1, intermediate, true, h1, hidden, true, intermediate, hidden, tokens, gw_1, hidden,
         true, "wgrad ffn1");
    ckrc(launch_colsum(dh1, tokens, intermediate, intermediate, gvec, s), "colsum");
    gemm(dh1, intermediate, false, w1, hidden, true, tokens, hidden, intermediate, da, hidden,
         false, "dgrad ffn1");
    ln_bwd(z1);
    gemm(dz, hidden, true, ctx, hidden, true, hidden, hidden, tokens, gw_o, hidden, true,
         "wgrad attn-out");
    gemm(dz, hidden, false, wo, hidden, true, tokens, hidden, hidden, dctx, hidden, false,
         "dgrad attn-out");
    {
      AttnArgs a;
      a.qkv = qkv; a.ctx = ctx; a.lse = lse; a.dctx = dctx; a.dqkv = dqkv; a.B = tokens / seq;
      a.S = seq; a.heads = heads; a.head_dim = head_dim;
      ckrc(launch_attention_bwd(a, s), "attention_bwd");
    }
    gemm(dqkv, 3 * hidden, true, x, hidden, true, 3 * hidden, hidden, tokens, gw_qkv, hidden,
         true, "wgrad qkv");
    ckrc(launch_colsum(dqkv, tokens, 3 * hidden, 3 * hidden, gvec, s), "colsum");
    gemm(dqkv, 3 * hidden, false, wqkv, hidden, true, tokens, hidden, 3 * hidden, dx, hidden,
         false, "dgrad qkv");
  };

  for (int i = 0; i < warmup; ++i) block();
  ck(cudaStreamSynchronize(s), "sync");
  ck(cudaEventRecord(e0, s), "record");
  for (int i = 0; i < iterations; ++i) {
    if (slowdown > 0) ckrc(launch_record_time(tslot, s), "record_time");
    block();
    // simulated slow device: spin on the GPU for slowdown x the block's own duration
    if (slowdown > 0) ckrc(launch_spin_factor(tslot, static_cast<float>(slowdown), s), "spin");
  }
  ck(cudaEventRecord(e1, s), "record");
  ck(cudaEventSynchronize(e1), "sync");
  float ms = 0.f;
  ck(cudaEventElapsedTime(&ms, e0, e1), "elapsed");

  for (void* p : allocs) cudaFree(p);
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(s);
  size_t free_b = 0, total_b = 0;
  ck(cudaMemGetInfo(&free_b, &total_b), "meminfo");
  return {static_cast<double>(ms) * 1e-3, static_cast<double>(free_b) / (1024.0 * 1024.0)};
}

}  // namespace sky
