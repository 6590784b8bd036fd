"""Multi-GPU pipeline check (run under torchrun): trains a small BERT for a few steps and prints
the per-step losses of the last stage as one JSON line, so that runs with different stage counts /
boundary transports / schedules can be compared (dropout is disabled => same math everywhere)."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import skycomputing_b200 as sky  # noqa: E402
from skycomputing_b200.models import BertConfig, set_backend  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--boundary", default="auto")
    ap.add_argument("--micro-batches", type=int, default=2)
    ap.add_argument("--layers", type=int, default=4)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--schedule", default="1f1b")
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--tag", default="")
    # attention heads of the hidden-1024 model: 16 = head size 64 (BERT-large), 8 = head size 128
    ap.add_argument("--heads", type=int, default=16)
    # > 1: looped pipeline (v chunks per GPU); add SKY_LOOPED_FUSED=1 for its fused ring boundary.
    # The loss trajectory must equal the plain pipeline's (same seeds per GLOBAL layer index).
    ap.add_argument("--virtual-stages", type=int, default=1)
    # "layer": the reference's granularity (cuts may fall after BertLayer_Head / Body)
    ap.add_argument("--granularity", default="block", choices=["block", "layer"])
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    set_backend("native")
    torch.manual_seed(7)
    cfg = BertConfig(30522, hidden_size=1024, num_hidden_layers=a.layers, num_attention_heads=a.heads,
                     intermediate_size=4096, hidden_dropout_prob=a.dropout,
                     attention_probs_dropout_prob=a.dropout)
    enc = [dict(layer_type="BertLayer_Head", config=cfg.__dict__),
           dict(layer_type="BertLayer_Body", config=cfg.__dict__),
           dict(layer_type="BertLayer_Tail", config=cfg.__dict__)] * a.layers
    model_config = ([dict(layer_type="BertEmbeddings", config=cfg.__dict__)] + enc
                    + [dict(layer_type="BertPooler", config=cfg.__dict__),
                       dict(layer_type="BertTailForClassification", hidden_dropout_prob=a.dropout,
                            hidden_size=1024, num_classes=3)])
    workers = [dict(name=f"gpu-{i}", server_config={}, device=i,
                    extra_config=dict(module_to_cuda=True, cuda_device=local, slowdown=0,
                                      mem_limit=-1, timer_config=dict(root="/tmp/sky_check")))
               for i in range(world)]
    wm = sky.WorkerManager(first_rank=0)
    wm.load_worker_pool_from_config(workers)
    wm = sky.Allocator(model_config, wm, granularity=a.granularity).allocate(
        "even", virtual_stages=a.virtual_stages)
    # identical initial weights regardless of the partition: seed per GLOBAL layer index
    model = sky.RpcModel(wm, this_rank=rank)
    for mod in model.model:
        if not mod.is_local:
            continue
        b0 = mod.layer_range[0]
        for off, layer in enumerate(mod.module.layers.children()):
            g = torch.Generator(device="cpu").manual_seed(1000 + b0 + off)
            with torch.no_grad():
                for p in layer.parameters():
                    p.copy_((torch.randn(p.shape, generator=g) * 0.02).to(p.device))
                for n, p in layer.named_parameters():
                    if n.endswith("LayerNorm.weight"):
                        p.fill_(1.0)
    opt = sky.build_optimizer(model.optim_module, dict(optim_type="SGD", lr=0.01))
    runner = sky.Runner(model=model, parameter_server=None, worker_manager=wm, optimizer=opt,
                        max_epochs=1, max_iters=10 ** 9, loss_cfg=dict(type="CrossEntropyLoss"),
                        timer_cfg=dict(root="/tmp/sky_check"), logging_cfg=None,
                        micro_batches=a.micro_batches, schedule=a.schedule, boundary=a.boundary,
                        use_cuda_graph=not a.no_graph, device=dev)
    model.train(True)
    ds = sky.SynthMNLIDataset(num_samples=a.batch * 2, max_seq_length=128, seed=3, full_length=False)
    losses = []
    for step in range(a.steps):
        sl = slice((step % 2) * a.batch, (step % 2 + 1) * a.batch)
        data = [ds.input_ids[sl], ds.segment_ids[sl], ds.input_mask[sl]]
        out = runner.train_iteration(data, ds.labels[sl])
        if out is not None:
            losses.append(round(out, 5))
    torch.cuda.synchronize()
    eng = runner.engine
    info = dict(tag=a.tag, world=world, boundary=a.boundary, schedule=eng.schedule,
                virtual_stages=a.virtual_stages, fused=(eng.in_fused or eng.out_fused),
                layers=[len(w.model_config) for w in wm.worker_pool],
                graph=eng._graph is not None, mb=a.micro_batches, losses=losses,
                err=eng.fused.error_code() if eng.fused is not None else 0)
    gathered = [None] * world
    dist.all_gather_object(gathered, info)
    if rank == 0:
        last = [g for g in gathered if g["losses"]][0]
        last["fused_any"] = any(g["fused"] for g in gathered)
        last["graph_all"] = all(g["graph"] for g in gathered)
        last["err_any"] = max(g["err"] for g in gathered)
        print("CHECK " + json.dumps(last), flush=True)
    eng.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
