// C++ device benchmark loop (the "stimulator benchmark" of the reference, re-done over device
// timers).  Reference: scaelum/dynamics/benchmarker.py:49-71 + estimator.py:15-34 time a Conv2d
// proxy with wall clock + cuda.synchronize and no warm-up; here every rank times the REAL kernel
// chain of a transformer block, forward AND backward (GEMMs, tcgen05 attention, LayerNorm,
// reductions: what BertSpanFn launches), with CUDA events after warm-up, so the measured speed
// predicts the real per-layer cost.
#pragma once
#include <utility>

namespace sky {
// returns (total seconds for `iterations` proxy blocks incl. simulated slowdown, free HBM in MiB)
// mode 0 = full forward + backward block (needs hidden == heads * head_dim, an attention shape
// the kernels support and tokens % seq == 0; falls back to mode 1 otherwise), mode 1 = the four
// forward GEMMs only
std::pair<double, double> device_benchmark(int tokens, int hidden, int intermediate, int iterations,
                                           int warmup, double slowdown, int mode = 0,
                                           int seq = 128, int heads = 16, int head_dim = 64);
}  // namespace sky
