"""Device and model benchmarkers (capability parity with scaelum/dynamics/benchmarker.py:30-201).

DeviceBenchmarker - "how fast is each device": in the SPMD design every rank benchmarks ITS OWN
GPU concurrently and the results are all-gathered (the reference pickles a 128 MiB input tensor
to every worker over RPC).  Two proxies:
  * ``proxy="model"`` (default, = reference): build ``model_config`` (e.g. 10 x Conv2d) as a
    stage and time ``iterations`` forwards (device-timed, optional warm-up);
  * ``proxy="bert_block"``: the C++ loop in csrc/bench/device_bench.cu times the real tcgen05
    GEMM chain of a transformer block with CUDA events, so the measured speed predicts the real
    per-layer cost.
The worker's ``slowdown`` is part of the measurement in both cases (device-side throttle), and
``STIMULATE=1`` applies the Stimulator multipliers (fixes the reference's broken import).

ModelBenchmarker - per-layer FLOPs / memory over the layer-config list.  Generic: identical
(config, input-signature) pairs are measured once and re-used, instead of the reference's
hard-coded BERT shortcut ``cfg[:4] + cfg[-2:]`` (benchmarker.py:163-166,197-201).
"""
from __future__ import annotations

import abc
import os
from typing import Dict, List, Optional

import torch

from ..builder import build_layer, build_module_from_cfg
from ..stimulator import Stimulator
from ..utils import generate_worker_name
from .estimator import Estimator
from .worker_manager import WorkerManager


class BaseBenchmarker(abc.ABC):
    @abc.abstractmethod
    def benchmark(self):
        raise NotImplementedError("not implemented yet")


def _dist_ready() -> bool:
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


class DeviceBenchmarker(BaseBenchmarker):
    def __init__(self, worker_manager: WorkerManager, data_generator, model_config: list,
                 iterations: int, dtype: Optional[str] = None, proxy: str = "model",
                 warmup: int = 0, block_shape: Optional[dict] = None):
        self._worker_manager = worker_manager
        self._model_config = model_config
        self._data_generator = data_generator
        self._iterations = iterations
        self._dtype = dtype
        self._proxy = proxy
        self._warmup = warmup
        self._block_shape = block_shape or dict(tokens=4096, hidden=1024, intermediate=4096)
        self._stimulator = (Stimulator(self._worker_manager.size)
                            if os.getenv("STIMULATE") is not None else None)

    @staticmethod
    def local_benchmark(rank, data, model_cfg, module_wrapper_cfg, iterations, dtype, warmup=0):
        """Build the proxy stage with the worker's own extra_config and time it."""
        cfg = dict(module_wrapper_cfg or {})
        cfg.pop("logging_config", None)  # benchmark runs must not write training logs
        model = build_module_from_cfg(rank=rank, model_cfg=model_cfg, module_wrapper_cfg=cfg)
        device = model.device
        t = Estimator.benchmark_speed(model=model, data=data, device=device,
                                      iterations=iterations, dtype=dtype, warmup=warmup)
        avai_mem = model.detect_mem(destroy_module=True)
        del model
        if torch.cuda.is_available():
            torch.cuda.empty_cache()
        return t, avai_mem

    @staticmethod
    def local_benchmark_native(module_wrapper_cfg, iterations, warmup, block_shape):
        from ..ops import native as nat

        cfg = module_wrapper_cfg or {}
        dev = cfg.get("cuda_device", -1)
        if dev is not None and dev >= 0:
            torch.cuda.set_device(dev)
        head_dim = int(block_shape.get("head_dim", 64))
        t, free_mib = nat.ext().device_benchmark(
            tokens=block_shape["tokens"], hidden=block_shape["hidden"],
            intermediate=block_shape["intermediate"], iterations=iterations,
            warmup=max(warmup, 1), slowdown=float(cfg.get("slowdown", 0) or 0),
            # the proxy is the block's real forward + backward kernel chain (GEMMs, attention,
            # LayerNorm, reductions); "gemm_only" selects round 1's four forward GEMMs
            mode=1 if block_shape.get("proxy_kernels") == "gemm_only" else 0,
            seq=int(block_shape.get("seq", 128)),
            heads=int(block_shape.get("heads", max(1, block_shape["hidden"] // head_dim))),
            head_dim=head_dim)
        mem_limit = cfg.get("mem_limit", -1)
        return t, (mem_limit if mem_limit and mem_limit > 0 else free_mib - 500)

    def _bench_worker(self, worker, data):
        if self._proxy == "bert_block":
            return self.local_benchmark_native(worker.extra_config, self._iterations, self._warmup,
                                               self._block_shape)
        return self.local_benchmark(worker.rank, data, self._model_config, worker.extra_config,
                                    self._iterations, self._dtype, self._warmup)

    def benchmark(self) -> Dict[str, dict]:
        import torch.distributed as dist

        pool = self._worker_manager.worker_pool
        data = self._data_generator.generate() if self._proxy == "model" else None
        measured: Dict[str, tuple] = {}
        if _dist_ready():
            me = dist.get_rank()
            mine = [w for w in pool if (w.device if w.device is not None else -1) == me]
            local = {w.name: self._bench_worker(w, data) for w in mine}
            gathered: List[dict] = [None] * dist.get_world_size()  # type: ignore[list-item]
            dist.all_gather_object(gathered, local)
            for part in gathered:
                measured.update(part)
        else:
            for w in pool:
                measured[w.name] = self._bench_worker(w, data)
        results: Dict[str, dict] = {}
        for w in pool:  # dict order = pool order (the allocator relies on it)
            t, avai_mem = measured[w.name]
            if self._stimulator is not None:
                t *= self._stimulator.compute_slowdown(w.rank)
                avai_mem /= self._stimulator.memory_slowdown(w.rank)
            results[generate_worker_name(w.rank)] = dict(time=t, avai_mem=avai_mem)
        return results


class ModelBenchmarker(BaseBenchmarker):
    def __init__(self, model_config: list, data_generator, device: str = "cpu",
                 dtype: Optional[str] = None, param_scale: int = 2, analytic: bool = False):
        self._analytic = analytic
        # stage boundaries carry bf16 on the native path (fp32 in the eager oracle / reference)
        self._boundary_elem_bytes = 2 if torch.cuda.is_available() else 4
        self._prev_out_bytes = 0.0
        self._model_config = model_config
        self._data_generator = data_generator
        self._device = device
        self._dtype = dtype
        self._param_scale = param_scale

    @property
    def model_config(self):
        return self._model_config

    @staticmethod
    def _signature(data) -> tuple:
        data = data if isinstance(data, (list, tuple)) else (data,)
        return tuple((tuple(d.shape), str(d.dtype)) if torch.is_tensor(d) else repr(d) for d in data)

    def benchmark(self):
        flops_list, mem_list = [], []
        # bytes_in[i] = what crosses a stage boundary placed IN FRONT of layer i (the floating
        # outputs of layer i - 1): feeds the allocator's comm-aware cut penalty
        self.last_boundary_bytes: List[float] = []
        data = self._data_generator.generate()
        cache: Dict[tuple, tuple] = {}
        for layer_cfg in self._model_config:
            key = (repr(sorted(layer_cfg.items(), key=lambda kv: kv[0])), self._signature(data))
            if key in cache:
                out_meta, flops, mem = cache[key]
                # re-materialise an output of the right shape without re-running the layer
                data = [torch.zeros(s, dtype=dt) for s, dt in out_meta]
            elif self._analytic and Estimator.analytic_layer_cost(layer_cfg, data) is not None:
                # closed-form FLOPs / memory for the registered BERT layers: no layer is built or
                # run (a 2 B-parameter model is costed in microseconds)
                flops, mem, out_meta = Estimator.analytic_layer_cost(layer_cfg, data,
                                                                     self._param_scale)
                cache[key] = (out_meta, flops, mem)
                data = [torch.zeros(s, dtype=dt) for s, dt in out_meta]
            else:
                cfg = dict(layer_cfg)
                layer = build_layer(cfg.pop("layer_type"), **cfg)
                output, flops, mem = Estimator.benchmark_model(
                    model=layer, data=data, device=self._device, dtype=self._dtype,
                    param_scale=self._param_scale)
                del layer
                outs = output if isinstance(output, (list, tuple)) else [output]
                outs = [o.detach().cpu() for o in outs]
                cache[key] = ([(tuple(o.shape), o.dtype) for o in outs], flops, mem)
                data = outs
            flops_list.append(flops)
            mem_list.append(mem)
            # payload in front of this layer = what the previous layer produced (set below)
            self.last_boundary_bytes.append(getattr(self, "_prev_out_bytes", 0.0))
            self._prev_out_bytes = float(sum(
                d.numel() * self._boundary_elem_bytes for d in data
                if torch.is_tensor(d) and d.is_floating_point()))
        self._prev_out_bytes = 0.0
        return flops_list, mem_list
