#!/usr/bin/env python
"""Headline benchmark: BERT-large training throughput (sequences/s, whole job) on N B200s.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by the driver as ``python -m torch.distributed.run --nproc-per-node N ...``
(one rank per GPU, RANK/LOCAL_RANK/WORLD_SIZE/MASTER_* from the env).  Workload = BASELINE.md §2:
BERT-large geometry (L=24, H=1024, A=16, I=4096, vocab 30522), MNLI-shaped batches (seq 128,
3 classes), SGD lr=1e-3, CrossEntropyLoss, dropout 0.1 active, synthetic data, random-init
weights.  Weak scaling: 32 sequences per GPU per step (global batch 32*N), layers split evenly
over the N pipeline stages by the framework's allocator.

Two timed regions, both bracketed by barrier + cuda.synchronize, max over ranks:
  value : K optimisation steps with the step's inputs already on the device (CUDA events);
  e2e   : K steps through the public API (Runner.train_iteration): every step copies its inputs
          from pinned host memory to the device and reads the loss back to the host.
Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEQ_LEN = 128
BATCH_PER_GPU = 32
LAYER_NUM = 24


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    # b1 = the reference's own layer classes + NCCL p2p (baseline/run_b1.py), fp32 or bf16-autocast
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "b1"])
    ap.add_argument("--b1-dtype", type=str, default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--b1-micro-batches", type=int, default=1)
    # `optimal` = the framework's exact load-balancing allocator over device benchmarks (the
    # capability under test); `even` is the reference's baseline split for comparison
    ap.add_argument("--alloc", type=str, default=os.environ.get("SKY_ALLOC", "optimal"),
                    choices=["even", "dynamic", "optimal"])
    ap.add_argument("--micro-batch", type=int, default=int(os.environ.get("SKY_MICRO_BATCH", "0")),
                    help="sequences per micro-batch (0 = auto)")
    ap.add_argument("--boundary", type=str, default=os.environ.get("SKY_BOUNDARY", "auto"))
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--layers", type=int, default=LAYER_NUM)
    # > 1: looped pipeline, v non-adjacent chunks per GPU on a ring of fused NVLink boundaries
    # (parallel/pipeline_looped.py); 0 = let the SchedulePlanner pick (micro-batch, count, v)
    ap.add_argument("--virtual-stages", type=int, default=int(os.environ.get("SKY_VIRTUAL_STAGES", "0")))
    ap.add_argument("--slow-rank", type=int, default=-1)
    ap.add_argument("--slowdown", type=float, default=0.0)
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the last timed step's loss and the updated parameters to DIR/*.npy")
    return ap.parse_args()


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._thr = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu_index)], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=3)
        sm = sorted(int(float(s[1])) for s in self.samples if len(s) > 2 and s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for name, val in zip(names, s[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def run_ours(args) -> dict:
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group(backend="nccl", rank=rank, world_size=world, device_id=device)

    from skycomputing_b200.models import set_backend
    from skycomputing_b200.ops import native as nat

    assert nat.available(), "sm_100a extension missing: run __graft_entry__.build()"
    set_backend("native")
    nat.enable_launch_counter()

    plan = pick_plan(args)
    result = measure(args, plan, rank, world, local_rank, device)
    if result == "fallback":
        # the planned schedule did not survive its warm-up (flag-wait error / non-finite loss on
        # some rank): measure the plain 1F1B pipeline instead and say so
        plain = dict(plan, virtual_stages=1, micro_batch=(BATCH_PER_GPU if args.gpus <= 2 else 16),
                     note="fallback from " + plan["schedule"])
        plain["micro_batches"] = BATCH_PER_GPU * args.gpus // plain["micro_batch"]
        plain["schedule"] = "1f1b"
        result = measure(args, plain, rank, world, local_rank, device)
        if result == "fallback":
            result = None
    b1 = measure_b1(args, world, rank)
    if result is not None and b1:
        result["vs_b1"] = {
            k: dict(b1_value=v["value"], b1_ms_per_step=v["ms_per_step"],
                    ratio=result["value"] / v["value"], b1_config=v["config"])
            for k, v in b1.items() if "value" in v}
        result["vs_b1"].update({k: v for k, v in b1.items() if "value" not in v})
        result["vs_b1"]["note"] = (
            "B1 = the reference's own layer classes + even split, NCCL send/recv boundaries "
            "(baseline/run_b1.py), measured in this process right after our timed region; "
            "bf16 = torch.autocast(bfloat16), the same-precision comparison for our bf16 kernels; "
            "fp32 = the reference's precision (our arm is bf16: not like for like)")
    dist.destroy_process_group()
    return result


def measure_b1(args, world, rank) -> dict:
    """Same-box B1 numbers for the `vs_b1` block, measured right after our timed region.

    B1 runs in a CHILD process group (its own torchrun) under a hard timeout: whatever the
    baseline does - including hanging in a mismatched send / recv - it cannot take our own
    measurement down.  Our ranks have released their engines and wait on the rendezvous store (no
    NCCL kernel spins on the GPUs meanwhile).  SKY_BENCH_B1=0 skips it."""
    if os.environ.get("SKY_BENCH_B1", "1") == "0":
        return {}
    import torch.distributed as dist

    N = args.gpus
    out = {}
    if rank == 0:
        env = {k: v for k, v in os.environ.items()
               if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_PORT", "GROUP_RANK",
                            "LOCAL_WORLD_SIZE", "ROLE_RANK", "ROLE_WORLD_SIZE", "TORCHELASTIC_RUN_ID")}
        port = int(os.environ.get("MASTER_PORT", "29533")) + 17
        for dtype, steps in (("bf16", 8), ("fp32", 4)):
            tail = [os.path.join(ROOT, "bench.py"), "--impl", "b1", "--gpus", str(N), "--steps",
                    str(steps), "--warmup", "3", "--b1-dtype", dtype, "--b1-micro-batches", str(N),
                    "--layers", str(args.layers)]
            if N > 1:
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                       f"--nproc-per-node={N}", "--master-addr", "127.0.0.1", "--master-port",
                       str(port)] + tail
            else:
                cmd = [sys.executable] + tail
            proc = None
            try:
                proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                                        text=True, env=env, start_new_session=True)
                stdout, _ = proc.communicate(timeout=150)
                line = [l for l in stdout.splitlines() if l.startswith("{")][-1]
                out[dtype] = json.loads(line)
            except subprocess.TimeoutExpired:
                import signal

                os.killpg(proc.pid, signal.SIGKILL)      # the session we started, nothing else
                proc.wait()
                out[dtype] = {"unavailable": "B1 timed out after 150 s"}
            except Exception as e:
                out[dtype] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
            port += 1
    if world > 1:
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("sky_b1_done", "1")
        else:
            from datetime import timedelta

            store.wait(["sky_b1_done"], timedelta(seconds=700))
    return out


def pick_plan(args) -> dict:
    """(micro-batch size, micro-batch count, virtual stages) for this GPU count.

    The SchedulePlanner's closed-form step model (dynamics/planner.py; it reproduced every measured
    multi-GPU step of round 1 within 2-8 %) ranks the candidates; per-stage costs are derived from
    the single-GPU step of the same per-GPU batch.  Flags / environment override the plan."""
    from skycomputing_b200.dynamics.planner import SchedulePlanner, costs_from_single_gpu_step

    N = args.gpus
    global_batch = BATCH_PER_GPU * N
    blocks_per_stage = max(1, args.layers // N)
    if args.slow_rank >= 0 and args.slowdown > 0 and args.alloc != "even":
        # heterogeneous devices: every GPU runs exactly v chunks of >= 1 block, so the allocator
        # can only shed work from a slow GPU if v leaves it room (v = blocks per GPU would pin
        # every GPU to its even share)
        blocks_per_stage = max(1, int(blocks_per_stage / (2.0 + args.slowdown)) or 1)
    single_gpu_step = 11.7e-3 * args.layers / 24.0      # measured: BENCH_r01 (32 sequences)
    planner = SchedulePlanner(N, costs_from_single_gpu_step(single_gpu_step, N), blocks_per_stage)
    sizes = (args.micro_batch,) if args.micro_batch else (16, 32)
    cands = planner.candidates(global_batch, micro_batch_sizes=sizes, allow_looped=N > 1)
    if args.virtual_stages > 0:
        cands = [c for c in cands if c.virtual_stages == args.virtual_stages] or cands
    # a looped pipeline needs at least as many micro-batches as ranks to keep the ring full
    cands = [c for c in cands if c.virtual_stages == 1 or c.micro_batches >= min(N, 2)] or cands
    best = cands[0]
    return dict(micro_batch=best.micro_batch, micro_batches=best.micro_batches,
                virtual_stages=best.virtual_stages if N > 1 else 1, schedule=best.schedule,
                predicted_ms=round(best.step_seconds * 1e3, 3))


def measure(args, plan, rank, world, local_rank, device):
    import torch
    import torch.distributed as dist

    import skycomputing_b200 as sky
    from skycomputing_b200.models import BertConfig
    from skycomputing_b200.ops import native as nat

    torch.manual_seed(1234)
    N = args.gpus
    global_batch = BATCH_PER_GPU * N
    mb = plan["micro_batch"]
    micro_batches = plan["micro_batches"]
    virtual_stages = plan["virtual_stages"]
    cfg = BertConfig.bert_large()
    encoder = [dict(layer_type="BertLayer_Head", config=cfg.__dict__),
               dict(layer_type="BertLayer_Body", config=cfg.__dict__),
               dict(layer_type="BertLayer_Tail", config=cfg.__dict__)] * args.layers
    model_config = ([dict(layer_type="BertEmbeddings", config=cfg.__dict__)] + encoder
                    + [dict(layer_type="BertPooler", config=cfg.__dict__),
                       dict(layer_type="BertTailForClassification",
                            hidden_dropout_prob=cfg.hidden_dropout_prob,
                            hidden_size=cfg.hidden_size, num_classes=3)])
    log_root = f"/tmp/sky_bench/{N}gpus"
    if rank == 0:
        os.makedirs(log_root, exist_ok=True)
    worker_config = [dict(name=f"gpu-{i}", server_config={}, device=i,
                          extra_config=dict(slowdown=args.slowdown if i == args.slow_rank else 0,
                                            mem_limit=-1, cuda_device=local_rank,
                                            module_to_cuda=True, output_to_cpu=False,
                                            timer_config=dict(root=log_root)))
                     for i in range(N)]
    wm = sky.WorkerManager(first_rank=0)
    wm.load_worker_pool_from_config(worker_config)

    model_bench = dev_bench = None
    if args.alloc != "even":
        gen = sky.build_data_generator("DataloaderGenerator", generator_cfg=dict(
            dataset_cfg=dict(type="SynthMNLIDataset", num_samples=mb, max_seq_length=SEQ_LEN),
            dataloader_cfg=dict(batch_size=mb)))
        model_bench = sky.ModelBenchmarker(model_config, gen, device="cpu", analytic=True)
        dev_bench = sky.DeviceBenchmarker(wm, None, model_config=[], iterations=20, warmup=3,
                                          proxy="bert_block",
                                          block_shape=dict(tokens=mb * SEQ_LEN, hidden=1024,
                                                           intermediate=4096))
    # `dynamic` = the greedy boundary-shifting solver (the reference's algorithm with its dead
    # shrink branch fixed), `optimal` = the exact min-max partition
    allocator = sky.Allocator(model_config, wm, model_bench, dev_bench, granularity="block",
                              solver="heuristic")
    wm = allocator.allocate(args.alloc, virtual_stages=virtual_stages if N > 1 else 1)
    layers_per_stage = [len(w.model_config) for w in wm.worker_pool]

    model = sky.RpcModel(wm, this_rank=rank)
    optimizer = sky.build_optimizer(model.optim_module, dict(optim_type="SGD", lr=1e-3))
    runner = sky.Runner(model=model, parameter_server=None, worker_manager=wm, optimizer=optimizer,
                        max_epochs=1, max_iters=10 ** 9, loss_cfg=dict(type="CrossEntropyLoss"),
                        timer_cfg=dict(root=log_root), logging_cfg=None,
                        micro_batches=micro_batches, schedule="1f1b" if micro_batches > 1 else "sequential",
                        boundary=args.boundary, use_cuda_graph=not args.no_graph, device=device,
                        async_loss=True)
    model.train(True)
    eng = runner.engine

    # synthetic MNLI-shaped batches in pinned host memory (one per step: no reuse across steps)
    total = args.warmup + args.steps
    ds = sky.SynthMNLIDataset(num_samples=global_batch * 4, max_seq_length=SEQ_LEN, seed=0)
    host_batches = []
    for i in range(4):
        sl = slice(i * global_batch, (i + 1) * global_batch)
        data = [ds.input_ids[sl].contiguous().pin_memory(), ds.segment_ids[sl].contiguous().pin_memory(),
                ds.input_mask[sl].contiguous().pin_memory()]
        host_batches.append((data, ds.labels[sl].contiguous().pin_memory()))
    dev_batches = [([t.to(device) for t in d], l.to(device)) for d, l in host_batches]

    def barrier_sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-timed region (inputs resident on the device) ----------------
    n_untimed = max(args.warmup, 5)  # >= 3 eager steps + graph capture happen in here
    warm_loss = None
    for i in range(n_untimed):
        d, l = dev_batches[i % 4]
        warm_loss = eng.train_step(d if eng.is_first else None, l if eng.is_last else None)
    barrier_sync()
    # health check of the schedule before anything is timed (all ranks agree on the verdict)
    bad = 0
    if eng.fused is not None and eng.fused.error_code():
        bad = 1
    if warm_loss is not None and not bool(torch.isfinite(warm_loss).all()):
        bad = 1
    if world > 1:
        bt = torch.tensor([bad], device=device)
        dist.all_reduce(bt, op=dist.ReduceOp.MAX)
        bad = int(bt.item())
    if bad:
        if rank == 0:
            print(f"[bench] plan {plan} failed its warm-up (flag error / non-finite loss)",
                  file=sys.stderr, flush=True)
        eng.close()
        del runner, model, optimizer, eng
        torch.cuda.empty_cache()
        return "fallback"
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    nat.reset_launch_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        d, l = dev_batches[i % 4]
        eng.train_step(d if eng.is_first else None, l if eng.is_last else None)
    e1.record()
    barrier_sync()
    dev_ms = e0.elapsed_time(e1)
    launches_eager = nat.launch_count()
    graph_launches = eng.launches_per_step * args.steps if eng._graph is not None else launches_eager
    # ---------------- end-to-end region through the public API ----------------
    for i in range(2):
        d, l = host_batches[i % 4]
        runner.train_iteration(d, l)
    barrier_sync()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    last_loss = None
    for i in range(args.steps):
        d, l = host_batches[i % 4]
        out = runner.train_iteration(d, l)
        last_loss = out if out is not None else last_loss
    out = runner.flush_loss()  # the last step's loss is read inside the timed region too
    last_loss = out if out is not None else last_loss
    e3.record()
    barrier_sync()
    e2e_ms = max(e2.elapsed_time(e3), (time.perf_counter() - t0) * 1e3)
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([dev_ms, e2e_ms, float(graph_launches)], device=device, dtype=torch.float64)
    if world > 1:
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone()
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, launches = tm[0].item(), tm[1].item(), int(ts[2].item())
        loss_t = torch.tensor([last_loss if last_loss is not None else -1.0], device=device)
        dist.all_reduce(loss_t, op=dist.ReduceOp.MAX)
        last_loss = loss_t.item()
    else:
        launches = int(graph_launches)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, model, last_loss, rank, world, device)
    err = eng.fused.error_code() if eng.fused is not None else 0
    # exposed stage-boundary communication (part of the BASELINE.json metric): per-crossing cost
    # of both fused boundary kernels, measured on ranks 0 / 1 right here, times the crossings a
    # rank has on its critical path per step
    boundary = None
    # (eng.fused is created collectively: the same verdict on every rank)
    if world > 1 and eng.fused is not None and os.environ.get("SKY_BENCH_BOUNDARY", "1") != "0":
        try:
            from skycomputing_b200.utils.boundary_probe import probe

            rows = probe(mb * SEQ_LEN)
            chunks = max(1, virtual_stages)
            per_cross = sum(r["exposed_us"] for r in rows.values())
            boundary = dict(
                exposed_boundary_ms_per_step=round(micro_batches * chunks * per_cross * 1e-3, 4),
                crossings_per_rank_and_step=micro_batches * chunks, per_crossing=rows,
                note="exposed = boundary kernel with peer stores + flags minus the same kernel "
                     "with local stores (CUDA-graph replays, both directions concurrently); "
                     "roofline = max(local compute, bytes / 900 GB/s)")
        except Exception as e:  # diagnostics must not take the measurement down
            boundary = dict(unavailable=f"{type(e).__name__}: {e}"[:200])
    if os.environ.get("SKY_TRACE", "0") == "1":
        _dump_trace(eng, rank, world, device, N)
    result = None
    n_params_m = 31.8 + 12.596 * args.layers + 1.05
    if rank == 0:
        value = global_batch * args.steps / (dev_ms * 1e-3)
        e2e = global_batch * args.steps / (e2e_ms * 1e-3)
        result = {
            "metric": "BERT-large training throughput (sequences/s, whole job)",
            "value": value, "unit": "sequences/s", "n_gpus": N, "steps": args.steps,
            "warmup": n_untimed, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "impl": "ours",
            "data": "synthetic MNLI-shaped (random ids, seq 128), random-init weights",
            "config": {
                "model": f"BERT-large L={args.layers} H=1024 A=16 I=4096 ({n_params_m:.0f}M params)",
                "global_batch": global_batch, "seq_len": SEQ_LEN,
                "parallelism": f"pp{N}" if N > 1 else "single-gpu",
                "micro_batches": micro_batches, "schedule": eng.schedule,
                "virtual_stages": getattr(model, "virtual_stages", 1),
                "allocator": args.alloc, "layers_per_stage": layers_per_stage,
                "plan": plan,
                "boundary": ("fused-nvlink-p2p" if (eng.in_fused or eng.out_fused) else
                             ("none" if N == 1 else "nccl-p2p")),
                "cuda_graph": eng._graph is not None, "optimizer": "fused SGD lr=1e-3, fp32 master weights",
                "dropout": 0.1,
                "l2": "no flush needed: per-step working set (2.0 GB weights+grads, >2 GB activations) "
                      ">> 126 MB L2; inputs rotate over 4 distinct batches",
            },
            "e2e": {"value": e2e, "unit": "sequences/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": 3 * global_batch * SEQ_LEN * 8 + global_batch * 8,
                    "d2h_bytes_per_step": 4,
                    "note": "Runner.train_iteration per step: H2D of the step's inputs from pinned "
                            "memory, graph replay, async D2H of the loss into pinned memory (read "
                            "by the host one step later; the last one before the timer stops)"},
            "gpu_launches": launches, "clocks": clocks, "final_loss": last_loss,
            "flag_wait_errors": err, "boundary": boundary,
        }
    eng.close()
    return result


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 128


def dump_outputs(out_dir, model, loss, rank, world, device):
    """--dump-outputs: what the timed path produced by its last step, as float32 .npy files: the
    mean loss (``loss.npy``) and every parameter after that step's SGD update
    (``param.<global layer index>.<parameter name>.npy``, so the files do not depend on how the
    layers were split over the GPUs).  A parameter larger than its share of the 64 MB budget is
    written as a fixed seeded sample of its elements, the same in every run, so that two builds
    run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    import torch.distributed as dist

    params = []
    for m in model.model:
        if m.is_local:
            first = m.layer_range[0] if m.layer_range else 0
            for i, layer in enumerate(m.module.layers.children()):
                params += [(f"param.{first + i:03d}.{n}", p) for n, p in layer.named_parameters()]
    n_files = torch.tensor([len(params)], device=device)
    if world > 1:
        dist.all_reduce(n_files)
    cap = (DUMP_LIMIT_BYTES // (int(n_files.item()) + 1) - NPY_HEADER_BYTES) // 4  # +1: loss.npy
    os.makedirs(out_dir, exist_ok=True)
    if rank == 0 and loss is not None:
        np.save(os.path.join(out_dir, "loss.npy"), np.asarray(loss, dtype=np.float32))
    for name, p in params:
        flat = p.detach().reshape(-1).float().cpu().numpy()
        if flat.size > cap:
            flat = flat[np.random.RandomState(0).randint(0, flat.size, cap)]
        np.save(os.path.join(out_dir, name + ".npy"), flat)


def _dump_trace(eng, rank, world, device, N):
    """SKY_TRACE=1: write the device timeline of the last step (tools/render_trace.py draws it).
    GPU %globaltimer clocks are aligned with barrier-bracketed stamps (median of 15)."""
    import json as _json

    import torch
    import torch.distributed as dist
    from skycomputing_b200.ops import native as nat

    slot = torch.zeros(1, dtype=torch.int64, device=device)
    offs = []
    for _ in range(15):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        nat.ext().record_time(slot.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        t = torch.tensor([slot.item()], dtype=torch.int64, device=device)
        if world > 1:
            g = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(g, t)
            offs.append(int(t.item() - g[0].item()))
        else:
            offs.append(0)
    offs.sort()
    out_dir = os.path.join(ROOT, "gpurun_out", "trace")
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"n{N}_rank{rank}.json"), "w") as f:
        _json.dump({"rank": rank, "stage": eng.s, "clock_offset_ns": offs[len(offs) // 2],
                    "events": [[list(tag), ns] for tag, ns in eng.trace()]}, f)


def main():
    args = parse_args()
    if args.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        try:
            import run_reference

            out = run_reference.run(args.gpus, args.steps, args.warmup, BATCH_PER_GPU, SEQ_LEN,
                                    args.layers)
        except Exception as e:  # the arm must never crash the driver
            import traceback

            traceback.print_exc()
            out = {"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"[:300]}
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(out), flush=True)
        return 0
    if args.impl == "b1":
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import run_b1

        out = run_b1.run(args.gpus, args.steps, args.warmup, args.b1_dtype, args.b1_micro_batches,
                         args.layers)
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(out), flush=True)
        return 0
    out = run_ours(args)
    if out is not None:
        print(json.dumps(out), flush=True)
    elif int(os.environ.get("RANK", "0")) == 0:
        # both the planned schedule and the plain 1F1B fallback failed their warm-up check
        print(json.dumps({"impl": "ours", "unavailable": "no schedule passed the warm-up health "
                          "check (flag-wait error or non-finite loss); see stderr"}), flush=True)
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
