// pybind11 bindings of the sm_100a kernel library + peer-memory (CUDA IPC) manager + the C++
// device benchmark loop.  Deliberately torch-free: tensors cross the boundary as raw device
// pointers (int) and the stream as `torch.cuda.current_stream().cuda_stream`, so this module
// builds in seconds and has no libtorch ABI coupling.  Python-side validation lives in
// skycomputing_b200/ops/.
#include <cuda_runtime.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "bench/device_bench.h"
#include "kernels/api.h"

namespace py = pybind11;
using sky::GemmArgs;

namespace {

template <class T>
T* P(uintptr_t v) {
  return reinterpret_cast<T*>(v);
}
cudaStream_t S(uintptr_t v) { return reinterpret_cast<cudaStream_t>(v); }

void check(int rc, const char* what) {
  if (rc != 0) {
    std::string msg = std::string(what) + " failed with code " + std::to_string(rc);
    if (rc > 0 && rc < 900) msg += std::string(" (") + cudaGetErrorString((cudaError_t)rc) + ")";
    throw std::runtime_error(msg);
  }
}
void cuda_check(cudaError_t e, const char* what) {
  if (e != cudaSuccess)
    throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

void gemm(uintptr_t A, uintptr_t B, int M, int N, int K, int lda, int ldb, bool a_mn, bool b_mn,
          uintptr_t out, int ldo, bool out_f32, bool accumulate, uintptr_t out2, int ldo2,
          uintptr_t bias, uintptr_t aux, int ldaux, int act, bool add_aux, float dropout_p,
          uintptr_t rng_state, uint32_t rng_stream, uintptr_t signal_flags, uintptr_t wait_flags,
          uintptr_t wait_epoch, uint32_t wait_mult, uintptr_t error_flag, int block_n, int pair, int stream_k, int max_ctas,
          int debug, uintptr_t ln_gamma, uintptr_t ln_beta, uintptr_t ln_mean, uintptr_t ln_rstd,
          float ln_eps,
          uintptr_t stream) {
  GemmArgs a;
  a.ln_gamma = P<const float>(ln_gamma);
  a.ln_beta = P<const float>(ln_beta);
  a.ln_mean = P<float>(ln_mean);
  a.ln_rstd = P<float>(ln_rstd);
  a.ln_eps = ln_eps;
  a.A = P<void>(A);
  a.B = P<void>(B);
  a.M = M;
  a.N = N;
  a.K = K;
  a.lda = lda;
  a.ldb = ldb;
  a.a_mn = a_mn;
  a.b_mn = b_mn;
  a.out = P<void>(out);
  a.ldo = ldo;
  a.out_f32 = out_f32;
  a.accumulate = accumulate;
  a.out2 = P<void>(out2);
  a.ldo2 = ldo2;
  a.bias = P<const float>(bias);
  a.aux = P<const void>(aux);
  a.ldaux = ldaux;
  a.act = act;
  a.add_aux = add_aux;
  a.dropout_p = dropout_p;
  a.rng_state = P<const uint64_t>(rng_state);
  a.rng_stream = rng_stream;
  a.signal_flags = P<uint32_t>(signal_flags);
  a.wait_flags = P<const uint32_t>(wait_flags);
  a.wait_epoch = P<const uint32_t>(wait_epoch);
  a.wait_mult = wait_mult;
  a.error_flag = P<int>(error_flag);
  a.block_n = block_n;
  a.pair = pair;
  a.stream_k = stream_k;
  a.max_ctas = max_ctas;
  a.debug = debug;
  check(sky::launch_gemm(a, S(stream)), "gemm");
}

void layernorm_fwd(uintptr_t z, uintptr_t y, uintptr_t mean, uintptr_t rstd, uintptr_t gamma,
                   uintptr_t beta, int M, int H, float eps, uintptr_t wait_flags,
                   uintptr_t wait_epoch, uint32_t wait_mult, uintptr_t error_flag,
                   uintptr_t signal_flags, uintptr_t stream) {
  sky::LayerNormFwdArgs a;
  a.signal_flags = P<uint32_t>(signal_flags);
  a.z = P<void>(z);
  a.y = P<void>(y);
  a.mean = P<float>(mean);
  a.rstd = P<float>(rstd);
  a.gamma = P<const float>(gamma);
  a.beta = P<const float>(beta);
  a.M = M;
  a.H = H;
  a.eps = eps;
  a.wait_flags = P<const uint32_t>(wait_flags);
  a.wait_epoch = P<const uint32_t>(wait_epoch);
  a.wait_mult = wait_mult;
  a.error_flag = P<int>(error_flag);
  check(sky::launch_layernorm_fwd(a, S(stream)), "layernorm_fwd");
}

void layernorm_bwd(uintptr_t dy, uintptr_t z, uintptr_t mean, uintptr_t rstd, uintptr_t gamma,
                   uintptr_t dz, uintptr_t dz_dropped, uintptr_t dgamma, uintptr_t dbeta, int M,
                   int H, float dropout_p, uintptr_t rng_state, uint32_t rng_stream,
                   uintptr_t wait_flags, uintptr_t wait_epoch, uint32_t wait_mult,
                   uintptr_t error_flag, uintptr_t stream) {
  sky::LayerNormBwdArgs a;
  a.dy = P<void>(dy);
  a.z = P<void>(z);
  a.mean = P<const float>(mean);
  a.rstd = P<const float>(rstd);
  a.gamma = P<const float>(gamma);
  a.dz = P<void>(dz);
  a.dz_dropped = P<void>(dz_dropped);
  a.dgamma = P<float>(dgamma);
  a.dbeta = P<float>(dbeta);
  a.M = M;
  a.H = H;
  a.dropout_p = dropout_p;
  a.rng_state = P<const uint64_t>(rng_state);
  a.rng_stream = rng_stream;
  a.wait_flags = P<const uint32_t>(wait_flags);
  a.wait_epoch = P<const uint32_t>(wait_epoch);
  a.wait_mult = wait_mult;
  a.error_flag = P<int>(error_flag);
  check(sky::launch_layernorm_bwd(a, S(stream)), "layernorm_bwd");
}

void colsum(uintptr_t x, int M, int N, int ldx, uintptr_t out, uintptr_t stream) {
  check(sky::launch_colsum(P<void>(x), M, N, ldx, P<float>(out), S(stream)), "colsum");
}

sky::AttnArgs make_attn(uintptr_t qkv, uintptr_t mask, uintptr_t ctx, uintptr_t lse,
                        uintptr_t dctx, uintptr_t dqkv, int B, int Sq, int heads, int head_dim, float scale,
                        float dropout_p, uintptr_t rng_state, uint32_t rng_stream) {
  sky::AttnArgs a;
  a.qkv = P<void>(qkv);
  a.mask = P<const float>(mask);
  a.ctx = P<void>(ctx);
  a.lse = P<float>(lse);
  a.dctx = P<void>(dctx);
  a.dqkv = P<void>(dqkv);
  a.B = B;
  a.S = Sq;
  a.heads = heads;
  a.head_dim = head_dim;
  a.scale = scale;
  a.dropout_p = dropout_p;
  a.rng_state = P<const uint64_t>(rng_state);
  a.rng_stream = rng_stream;
  return a;
}
void attention_fwd(uintptr_t qkv, uintptr_t mask, uintptr_t ctx, uintptr_t lse, int B, int Sq, int heads,
                   int head_dim, float scale, float dropout_p, uintptr_t rng_state,
                   uint32_t rng_stream, uintptr_t stream) {
  auto a = make_attn(qkv, mask, ctx, lse, 0, 0, B, Sq, heads, head_dim, scale, dropout_p, rng_state,
                     rng_stream);
  check(sky::launch_attention_fwd(a, S(stream)), "attention_fwd");
}
void attention_bwd(uintptr_t qkv, uintptr_t mask, uintptr_t ctx, uintptr_t lse, uintptr_t dctx,
                   uintptr_t dqkv, int B, int Sq,
                   int heads, int head_dim, float scale, float dropout_p, uintptr_t rng_state,
                   uint32_t rng_stream, uintptr_t stream) {
  auto a = make_attn(qkv, mask, ctx, lse, dctx, dqkv, B, Sq, heads, head_dim, scale, dropout_p,
                     rng_state, rng_stream);
  check(sky::launch_attention_bwd(a, S(stream)), "attention_bwd");
}

void embed_fwd(uintptr_t ids, uintptr_t tts, uintptr_t amask, uintptr_t word, uintptr_t pos,
               uintptr_t type, uintptr_t gamma, uintptr_t beta, uintptr_t out, uintptr_t ext_mask,
               uintptr_t mean, uintptr_t rstd, int B, int Sq, int H, float eps, float dropout_p,
               uintptr_t rng_state, uint32_t rng_stream, uintptr_t stream) {
  sky::EmbedArgs a;
  a.input_ids = P<const int64_t>(ids);
  a.token_type = P<const int64_t>(tts);
  a.attn_mask = P<const int64_t>(amask);
  a.word = P<const float>(word);
  a.pos = P<const float>(pos);
  a.type = P<const float>(type);
  a.gamma = P<const float>(gamma);
  a.beta = P<const float>(beta);
  a.out = P<void>(out);
  a.ext_mask = P<float>(ext_mask);
  a.mean = P<float>(mean);
  a.rstd = P<float>(rstd);
  a.B = B;
  a.S = Sq;
  a.H = H;
  a.eps = eps;
  a.dropout_p = dropout_p;
  a.rng_state = P<const uint64_t>(rng_state);
  a.rng_stream = rng_stream;
  check(sky::launch_embed_fwd(a, S(stream)), "embed_fwd");
}

void embed_bwd(uintptr_t dout, uintptr_t ids, uintptr_t tts, uintptr_t word, uintptr_t pos,
               uintptr_t type, uintptr_t gamma, uintptr_t mean, uintptr_t rstd, uintptr_t dword,
               uintptr_t dpos, uintptr_t dtype_, uintptr_t dgamma, uintptr_t dbeta, int B, int Sq,
               int H, float dropout_p, uintptr_t rng_state, uint32_t rng_stream,
               uintptr_t wait_flags, uintptr_t wait_epoch, uint32_t wait_mult,
               uintptr_t error_flag, int type_rows, uintptr_t stream) {
  sky::EmbedBwdArgs a;
  a.type_rows = type_rows;
  a.dout = P<void>(dout);
  a.input_ids = P<const int64_t>(ids);
  a.token_type = P<const int64_t>(tts);
  a.word = P<const float>(word);
  a.pos = P<const float>(pos);
  a.type = P<const float>(type);
  a.gamma = P<const float>(gamma);
  a.mean = P<const float>(mean);
  a.rstd = P<const float>(rstd);
  a.dword = P<float>(dword);
  a.dpos = P<float>(dpos);
  a.dtype_ = P<float>(dtype_);
  a.dgamma = P<float>(dgamma);
  a.dbeta = P<float>(dbeta);
  a.B = B;
  a.S = Sq;
  a.H = H;
  a.dropout_p = dropout_p;
  a.rng_state = P<const uint64_t>(rng_state);
  a.rng_stream = rng_stream;
  a.wait_flags = P<const uint32_t>(wait_flags);
  a.wait_epoch = P<const uint32_t>(wait_epoch);
  a.wait_mult = wait_mult;
  a.error_flag = P<int>(error_flag);
  check(sky::launch_embed_bwd(a, S(stream)), "embed_bwd");
}

void small_linear_fwd(uintptr_t x, bool x_bf16, int ldx, uintptr_t w, uintptr_t b, uintptr_t y,
                      int M, int N, int K, int act_tanh, float dropout_p, uintptr_t rng_state,
                      uint32_t rng_stream, uintptr_t stream) {
  check(sky::launch_small_linear_fwd(P<void>(x), x_bf16, ldx, P<const float>(w),
                                     P<const float>(b), P<float>(y), M, N, K, act_tanh, dropout_p,
                                     P<const uint64_t>(rng_state), rng_stream, S(stream)),
        "small_linear_fwd");
}
void small_linear_bwd(uintptr_t x, bool x_bf16, int ldx, uintptr_t w, uintptr_t y, uintptr_t dy,
                      uintptr_t dx, bool dx_bf16, int lddx, uintptr_t dw, uintptr_t db, int M,
                      int N, int K, int act_tanh, float dropout_p, uintptr_t rng_state,
                      uint32_t rng_stream, uintptr_t stream) {
  check(sky::launch_small_linear_bwd(P<void>(x), x_bf16, ldx, P<const float>(w),
                                     P<const float>(y), P<const float>(dy), P<void>(dx), dx_bf16,
                                     lddx, P<float>(dw), P<float>(db), M, N, K, act_tanh,
                                     dropout_p, P<const uint64_t>(rng_state), rng_stream,
                                     S(stream)),
        "small_linear_bwd");
}
void softmax_ce(uintptr_t logits, uintptr_t labels, uintptr_t loss, uintptr_t dlogits, int M,
                int C, float grad_scale, uintptr_t loss_acc, uintptr_t stream) {
  check(sky::launch_softmax_ce(P<const float>(logits), P<const int64_t>(labels), P<float>(loss),
                               P<float>(dlogits), M, C, grad_scale, P<float>(loss_acc), S(stream)),
        "softmax_ce");
}

// descriptors: list of (p, g, mom, p_bf16, numel) -> packed host bytes to upload once
py::bytes pack_sgd_descriptors(
    const std::vector<std::tuple<uintptr_t, uintptr_t, uintptr_t, uintptr_t, long long, int,
                                 uintptr_t>>& ts) {
  std::vector<sky::SgdTensor> v(ts.size());
  for (size_t i = 0; i < ts.size(); ++i) {
    v[i].p = P<float>(std::get<0>(ts[i]));
    v[i].g = P<float>(std::get<1>(ts[i]));
    v[i].mom = P<float>(std::get<2>(ts[i]));
    v[i].p_bf16 = P<void>(std::get<3>(ts[i]));
    v[i].numel = std::get<4>(ts[i]);
    v[i].skip_zero = std::get<5>(ts[i]);
    v[i].pad_ = 0;
    v[i].mom2 = P<float>(std::get<6>(ts[i]));
  }
  return py::bytes(reinterpret_cast<const char*>(v.data()), v.size() * sizeof(sky::SgdTensor));
}
void sgd_multi(uintptr_t d_tensors, int n, long long max_numel, float lr, float momentum,
               float weight_decay, float grad_scale, bool zero_grad, uintptr_t stream) {
  check(sky::launch_sgd_multi(P<const sky::SgdTensor>(d_tensors), n, max_numel, lr, momentum,
                              weight_decay, grad_scale, zero_grad, S(stream)),
        "sgd_multi");
}
void adam_multi(uintptr_t d_tensors, int n, long long max_numel, float lr, float beta1, float beta2,
                float eps, float weight_decay, bool decoupled, uintptr_t step, float grad_scale,
                bool zero_grad, uintptr_t stream) {
  check(sky::launch_adam_multi(P<const sky::SgdTensor>(d_tensors), n, max_numel, lr, beta1, beta2,
                               eps, weight_decay, decoupled, P<const uint64_t>(step), grad_scale,
                               zero_grad, S(stream)),
        "adam_multi");
}
void cast_f32_to_bf16(uintptr_t src, uintptr_t dst, long long n, uintptr_t stream) {
  check(sky::launch_cast_f32_to_bf16(P<const float>(src), P<void>(dst), n, S(stream)), "cast");
}
void cast_bf16_to_f32(uintptr_t src, uintptr_t dst, long long n, uintptr_t stream) {
  check(sky::launch_cast_bf16_to_f32(P<const void>(src), P<float>(dst), n, S(stream)), "cast");
}

// ----------------------------------------------------------------------------------------------
// peer memory (CUDA IPC): buffers + flags that live in THIS process' HBM and are mapped by peers
// ----------------------------------------------------------------------------------------------
std::pair<uintptr_t, py::bytes> ipc_alloc(size_t nbytes) {
  void* p = nullptr;
  cuda_check(cudaMalloc(&p, nbytes), "cudaMalloc");
  cuda_check(cudaMemset(p, 0, nbytes), "cudaMemset");
  cudaIpcMemHandle_t h;
  cuda_check(cudaIpcGetMemHandle(&h, p), "cudaIpcGetMemHandle");
  return {reinterpret_cast<uintptr_t>(p),
          py::bytes(reinterpret_cast<const char*>(&h), sizeof(h))};
}
uintptr_t ipc_open(const std::string& handle) {
  if (handle.size() != sizeof(cudaIpcMemHandle_t)) throw std::runtime_error("bad ipc handle");
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle.data(), sizeof(h));
  void* p = nullptr;
  cuda_check(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
  return reinterpret_cast<uintptr_t>(p);
}
void ipc_close(uintptr_t p) { cuda_check(cudaIpcCloseMemHandle(P<void>(p)), "ipc_close"); }
void dev_free(uintptr_t p) { cuda_check(cudaFree(P<void>(p)), "cudaFree"); }
uintptr_t dev_malloc(size_t nbytes) {
  void* p = nullptr;
  cuda_check(cudaMalloc(&p, nbytes), "cudaMalloc");
  cuda_check(cudaMemset(p, 0, nbytes), "cudaMemset");
  return reinterpret_cast<uintptr_t>(p);
}
bool enable_peer_access(int peer) {
  int can = 0, dev = 0;
  cuda_check(cudaGetDevice(&dev), "cudaGetDevice");
  if (peer == dev) return true;
  cuda_check(cudaDeviceCanAccessPeer(&can, dev, peer), "cudaDeviceCanAccessPeer");
  if (!can) return false;
  cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    return true;
  }
  cuda_check(e, "cudaDeviceEnablePeerAccess");
  return true;
}
void memset_async(uintptr_t p, int value, size_t nbytes, uintptr_t stream) {
  cuda_check(cudaMemsetAsync(P<void>(p), value, nbytes, S(stream)), "cudaMemsetAsync");
}
void memcpy_h2d(uintptr_t dst, const std::string& src, uintptr_t stream) {
  cuda_check(cudaMemcpyAsync(P<void>(dst), src.data(), src.size(), cudaMemcpyHostToDevice,
                             S(stream)),
             "memcpy_h2d");
  cuda_check(cudaStreamSynchronize(S(stream)), "sync");
}
py::bytes memcpy_d2h(uintptr_t src, size_t nbytes) {
  std::string buf(nbytes, '\0');
  cuda_check(cudaMemcpy(buf.data(), P<void>(src), nbytes, cudaMemcpyDeviceToHost), "memcpy_d2h");
  return py::bytes(buf);
}
std::pair<size_t, size_t> mem_info() {
  size_t f = 0, t = 0;
  cuda_check(cudaMemGetInfo(&f, &t), "cudaMemGetInfo");
  return {f, t};
}

}  // namespace

PYBIND11_MODULE(_cuda, m) {
  m.doc() = "skycomputing_b200 sm_100a kernel library";
  m.def("gemm", &gemm, py::arg("A"), py::arg("B"), py::arg("M"), py::arg("N"), py::arg("K"),
        py::arg("lda"), py::arg("ldb"), py::arg("a_mn") = false, py::arg("b_mn") = false,
        py::arg("out"), py::arg("ldo"), py::arg("out_f32") = false, py::arg("accumulate") = false,
        py::arg("out2") = 0, py::arg("ldo2") = 0, py::arg("bias") = 0, py::arg("aux") = 0,
        py::arg("ldaux") = 0, py::arg("act") = 0, py::arg("add_aux") = false,
        py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0, py::arg("rng_stream") = 0,
        py::arg("signal_flags") = 0, py::arg("wait_flags") = 0, py::arg("wait_epoch") = 0,
        py::arg("wait_mult") = 0, py::arg("error_flag") = 0, py::arg("block_n") = 0, py::arg("pair") = -1, py::arg("stream_k") = -1,
        py::arg("max_ctas") = 0, py::arg("debug") = 0, py::arg("ln_gamma") = 0,
        py::arg("ln_beta") = 0, py::arg("ln_mean") = 0, py::arg("ln_rstd") = 0,
        py::arg("ln_eps") = 1e-12f, py::arg("stream") = 0);
  m.def("attention_supported", &sky::attention_supported, py::arg("S"), py::arg("head_dim"));
  m.def("gemm_ln_block_n", &sky::gemm_ln_block_n, py::arg("M"), py::arg("N"),
        py::arg("force") = false);
  m.def("gemm_ln_tiles_per_panel", &sky::gemm_ln_tiles_per_panel, py::arg("M"), py::arg("N"),
        py::arg("force") = false);
  m.def("gemm_pick_block_n", &sky::gemm_pick_block_n);
  m.def("gemm_tiles_per_panel", &sky::gemm_tiles_per_panel);
  m.def("layernorm_fwd", &layernorm_fwd, py::arg("z"), py::arg("y"), py::arg("mean"),
        py::arg("rstd"), py::arg("gamma"), py::arg("beta"), py::arg("M"), py::arg("H"),
        py::arg("eps"), py::arg("wait_flags") = 0, py::arg("wait_epoch") = 0,
        py::arg("wait_mult") = 0, py::arg("error_flag") = 0, py::arg("signal_flags") = 0,
        py::arg("stream") = 0);
  m.attr("LN_SIGNALS_PER_PANEL") = sky::kLnSignalsPerPanel;
  m.def("dgelu_mul", [](uintptr_t g, uintptr_t h, uintptr_t y, long long n, uintptr_t s) {
    check(sky::launch_dgelu_mul(P<const void>(g), P<const void>(h), P<void>(y), n, S(s)),
          "dgelu_mul");
  });
  m.def("layernorm_bwd", &layernorm_bwd, py::arg("dy"), py::arg("z"), py::arg("mean"),
        py::arg("rstd"), py::arg("gamma"), py::arg("dz"), py::arg("dz_dropped") = 0,
        py::arg("dgamma"), py::arg("dbeta"), py::arg("M"), py::arg("H"),
        py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0, py::arg("rng_stream") = 0,
        py::arg("wait_flags") = 0, py::arg("wait_epoch") = 0, py::arg("wait_mult") = 0,
        py::arg("error_flag") = 0, py::arg("stream") = 0);
  m.def("ln_param_grad", [](uintptr_t dy, uintptr_t z, uintptr_t mean, uintptr_t rstd,
                            uintptr_t dgamma, uintptr_t dbeta, int M, int H, uintptr_t x2,
                            uintptr_t out2, uintptr_t stream) {
    check(sky::launch_ln_param_grad(P<void>(dy), P<void>(z), P<const float>(mean),
                                    P<const float>(rstd), P<float>(dgamma), P<float>(dbeta), M, H,
                                    P<void>(x2), P<float>(out2), S(stream)),
          "ln_param_grad");
  }, py::arg("dy"), py::arg("z"), py::arg("mean"), py::arg("rstd"), py::arg("dgamma"),
        py::arg("dbeta"), py::arg("M"), py::arg("H"), py::arg("x2") = 0, py::arg("out2") = 0,
        py::arg("stream") = 0);
  m.def("colsum", &colsum, py::arg("x"), py::arg("M"), py::arg("N"), py::arg("ldx"),
        py::arg("out"), py::arg("stream") = 0);
  m.def("attention_fwd", &attention_fwd, py::arg("qkv"), py::arg("mask"), py::arg("ctx"),
        py::arg("lse"), py::arg("B"), py::arg("S"), py::arg("heads"), py::arg("head_dim"), py::arg("scale"),
        py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0, py::arg("rng_stream") = 0,
        py::arg("stream") = 0);
  m.def("attention_bwd", &attention_bwd, py::arg("qkv"), py::arg("mask"), py::arg("ctx"),
        py::arg("lse"), py::arg("dctx"), py::arg("dqkv"), py::arg("B"), py::arg("S"), py::arg("heads"), py::arg("head_dim"),
        py::arg("scale"), py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0,
        py::arg("rng_stream") = 0, py::arg("stream") = 0);
  m.def("embed_fwd", &embed_fwd, py::arg("ids"), py::arg("tts"), py::arg("amask"),
        py::arg("word"), py::arg("pos"), py::arg("type"), py::arg("gamma"), py::arg("beta"),
        py::arg("out"), py::arg("ext_mask"), py::arg("mean"), py::arg("rstd"), py::arg("B"),
        py::arg("S"), py::arg("H"), py::arg("eps"), py::arg("dropout_p") = 0.f,
        py::arg("rng_state") = 0, py::arg("rng_stream") = 0, py::arg("stream") = 0);
  m.def("embed_bwd", &embed_bwd, py::arg("dout"), py::arg("ids"), py::arg("tts"), py::arg("word"),
        py::arg("pos"), py::arg("type"), py::arg("gamma"), py::arg("mean"), py::arg("rstd"),
        py::arg("dword"), py::arg("dpos"), py::arg("dtype"), py::arg("dgamma"), py::arg("dbeta"),
        py::arg("B"), py::arg("S"), py::arg("H"), py::arg("dropout_p") = 0.f,
        py::arg("rng_state") = 0, py::arg("rng_stream") = 0, py::arg("wait_flags") = 0,
        py::arg("wait_epoch") = 0, py::arg("wait_mult") = 0, py::arg("error_flag") = 0,
        py::arg("type_rows") = 2, py::arg("stream") = 0);
  m.def("small_linear_fwd", &small_linear_fwd, py::arg("x"), py::arg("x_bf16"), py::arg("ldx"),
        py::arg("w"), py::arg("b"), py::arg("y"), py::arg("M"), py::arg("N"), py::arg("K"),
        py::arg("act_tanh") = 0, py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0,
        py::arg("rng_stream") = 0, py::arg("stream") = 0);
  m.def("small_linear_bwd", &small_linear_bwd, py::arg("x"), py::arg("x_bf16"), py::arg("ldx"),
        py::arg("w"), py::arg("y"), py::arg("dy"), py::arg("dx"), py::arg("dx_bf16"),
        py::arg("lddx"), py::arg("dw"), py::arg("db"), py::arg("M"), py::arg("N"), py::arg("K"),
        py::arg("act_tanh") = 0, py::arg("dropout_p") = 0.f, py::arg("rng_state") = 0,
        py::arg("rng_stream") = 0, py::arg("stream") = 0);
  m.def("softmax_ce", &softmax_ce, py::arg("logits"), py::arg("labels"), py::arg("loss"),
        py::arg("dlogits"), py::arg("M"), py::arg("C"), py::arg("grad_scale") = 1.f,
        py::arg("loss_acc") = 0, py::arg("stream") = 0);
  m.def("pack_sgd_descriptors", &pack_sgd_descriptors);
  m.def("sgd_multi", &sgd_multi, py::arg("d_tensors"), py::arg("n"), py::arg("max_numel"),
        py::arg("lr"), py::arg("momentum") = 0.f, py::arg("weight_decay") = 0.f,
        py::arg("grad_scale") = 1.f, py::arg("zero_grad") = true, py::arg("stream") = 0);
  m.def("adam_multi", &adam_multi, py::arg("d_tensors"), py::arg("n"), py::arg("max_numel"),
        py::arg("lr"), py::arg("beta1") = 0.9f, py::arg("beta2") = 0.999f, py::arg("eps") = 1e-8f,
        py::arg("weight_decay") = 0.f, py::arg("decoupled") = false, py::arg("step") = 0,
        py::arg("grad_scale") = 1.f, py::arg("zero_grad") = true, py::arg("stream") = 0);
  m.def("cast_f32_to_bf16", &cast_f32_to_bf16);
  m.def("cast_bf16_to_f32", &cast_bf16_to_f32);

  m.def("advance_counter", [](uintptr_t c, uint64_t inc, uintptr_t s) {
    check(sky::launch_advance_counter(P<uint64_t>(c), inc, S(s)), "advance_counter");
  });
  m.def("advance_epoch", [](uintptr_t c, uint32_t inc, uintptr_t s) {
    check(sky::launch_advance_epoch(P<uint32_t>(c), inc, S(s)), "advance_epoch");
  });
  m.def("signal_flags", [](uintptr_t f, int n, uint32_t inc, uintptr_t s) {
    check(sky::launch_signal_flags(P<uint32_t>(f), n, inc, S(s)), "signal_flags");
  });
  m.def("wait_flags", [](uintptr_t f, int n, uintptr_t epoch, uint32_t mult, uintptr_t err,
                         uintptr_t s) {
    check(sky::launch_wait_flags(P<const uint32_t>(f), n, P<const uint32_t>(epoch), mult,
                                 P<int>(err), S(s)),
          "wait_flags");
  });
  m.def("spin_ns", [](uint64_t ns, uintptr_t s) {
    check(sky::launch_spin_ns(ns, S(s)), "spin_ns");
  });
  m.def("record_time", [](uintptr_t slot, uintptr_t s) {
    check(sky::launch_record_time(P<uint64_t>(slot), S(s)), "record_time");
  });
  m.def("spin_factor", [](uintptr_t slot, float factor, uintptr_t s) {
    check(sky::launch_spin_factor(P<const uint64_t>(slot), factor, S(s)), "spin_factor");
  });
  m.def("peer_copy_signal", [](uintptr_t src, uintptr_t dst, long long nbytes, uintptr_t flags,
                               int n_flags, uint32_t inc, uintptr_t s) {
    check(sky::launch_peer_copy_signal(P<const void>(src), P<void>(dst), nbytes,
                                       P<uint32_t>(flags), n_flags, inc, S(s)),
          "peer_copy_signal");
  });

  m.def("ipc_alloc", &ipc_alloc);
  m.def("ipc_open", &ipc_open);
  m.def("ipc_close", &ipc_close);
  m.def("dev_malloc", &dev_malloc);
  m.def("dev_free", &dev_free);
  m.def("enable_peer_access", &enable_peer_access);
  m.def("memset_async", &memset_async);
  m.def("memcpy_h2d", &memcpy_h2d);
  m.def("memcpy_d2h", &memcpy_d2h);
  m.def("mem_info", &mem_info);

  m.def("device_benchmark", &sky::device_benchmark, py::arg("tokens"), py::arg("hidden"),
        py::arg("intermediate"), py::arg("iterations"), py::arg("warmup"),
        py::arg("slowdown") = 0.0, py::arg("mode") = 0, py::arg("seq") = 128,
        py::arg("heads") = 16, py::arg("head_dim") = 64,
        "C++ device benchmark loop: times `iterations` transformer blocks (mode 0: the full "
        "forward + backward kernel chain, mode 1: forward GEMMs only) with CUDA events; returns "
        "(seconds_total, free_mem_MiB)");
}
