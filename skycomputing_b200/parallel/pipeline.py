"""SPMD pipeline engine: one process per GPU, each owning one contiguous layer span.

What the reference does with RPC (scaelum/model/rpc_model.py:44-55, runner.py:127-139: the master
issues one remote forward per stage, stages pull activations through CPU, distributed autograd
walks back, a DistributedOptimizer steps every owner) happens here inside every rank:

    for each micro-batch (sequential or 1F1B order):
        obtain the stage input  (own data | fused peer slot | NCCL/gloo recv)
        run the stage           (ModuleWrapper -> fused sm_100a spans)
        hand the output on      (LayerNorm wrote it into the next GPU already | send)
        ... backward symmetric  (dgrad GEMM writes into the previous GPU | send)
    optimizer step              (FusedSGD: one launch)

Boundaries are FUSED (parallel/p2p.py) when the cut sits between two whole transformer blocks on
the native path, and fall back to torch.distributed p2p (nccl / gloo) otherwise.  When every link
of a rank is fused (or absent) the whole step - all micro-batches, backward, optimizer, RNG/epoch
counters - is captured into ONE CUDA graph and replayed; cross-GPU synchronisation then happens
exclusively through in-kernel flag waits.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import torch
import torch.distributed as dist

from ..builder.module_wrapper import ModuleWrapper
from ..ops.native import attention_supported
from .engine_base import EngineBase


def one_f_one_b_order(stage: int, num_stages: int, micro_batches: int) -> List[tuple]:
    """[('F', j) | ('B', j)] for this stage (non-interleaved 1F1B)."""
    warm = min(num_stages - stage - 1, micro_batches)
    order: List[tuple] = [("F", j) for j in range(warm)]
    f, b = warm, 0
    for _ in range(micro_batches - warm):
        order.append(("F", f))
        f += 1
        order.append(("B", b))
        b += 1
    while b < micro_batches:
        order.append(("B", b))
        b += 1
    return order


def sequential_order(stage: int, num_stages: int, micro_batches: int) -> List[tuple]:
    """One micro-batch in flight at a time (reference semantics when micro_batches == 1)."""
    order: List[tuple] = []
    for j in range(micro_batches):
        order += [("F", j), ("B", j)]
    return order


class PipelineEngine(EngineBase):
    def __init__(self, stage: ModuleWrapper, stage_index: int, num_stages: int,
                 stage_to_rank: Sequence[int], device: torch.device, optimizer,
                 loss_fn: Optional[Callable] = None, micro_batches: int = 1,
                 schedule: str = "1f1b", boundary: str = "auto", use_cuda_graph: bool = True,
                 group=None, advance_rng: bool = True):
        assert schedule in ("1f1b", "sequential"), schedule
        assert boundary in ("auto", "fused", "nccl", "gloo", "dist"), boundary
        self.stage = stage
        self.s, self.P = stage_index, num_stages
        self.stage_to_rank = list(stage_to_rank)
        self.device = device
        self.optimizer = optimizer
        self.loss_fn = loss_fn
        self.m = micro_batches
        self.schedule = schedule
        self.boundary = boundary
        self.group = group
        self.is_first, self.is_last = stage_index == 0, stage_index == num_stages - 1
        self.prev_rank = None if self.is_first else self.stage_to_rank[stage_index - 1]
        self.next_rank = None if self.is_last else self.stage_to_rank[stage_index + 1]
        self.comm = None
        self.fused = None
        self.in_fused = self.out_fused = False
        self._setup_done = False
        self._want_graph = use_cuda_graph and device.type == "cuda"
        self._graph = None
        self._static_inputs: Optional[list] = None
        self._static_labels: Optional[torch.Tensor] = None
        self._loss_acc: Optional[torch.Tensor] = None
        self._eager_steps = 0
        self._advance_rng = advance_rng
        self._pending_sends: list = []
        self.stage.engine_managed_backward = True
        self.launches_per_step = 0
        self._init_common()

    # ------------------------------------------------------------------ setup
    def _setup(self, inputs: Optional[Sequence[torch.Tensor]]) -> None:
        multi = self.P > 1
        shape = [0, 0]
        if multi:
            if self.is_first:
                b = inputs[0].shape[0]
                shape = [b // self.m, int(inputs[0].shape[1]) if inputs[0].dim() > 1 else 0]
            obj = [shape]
            dist.broadcast_object_list(obj, src=self.stage_to_rank[0], group=self.group)
            shape = obj[0]
        elif inputs is not None:
            shape = [inputs[0].shape[0] // self.m, int(inputs[0].shape[1]) if inputs[0].dim() > 1 else 0]
        self.mb_batch, self.seq = shape
        want_fused = self.boundary in ("auto", "fused") and self._native_active() and multi
        in_ok = out_ok = False
        hidden = 0
        if want_fused:
            spans = self.stage.spans()
            if spans:
                hidden = self._hidden_size(spans[0])
            in_ok, out_ok = self.stage.fused_boundary_support((self.mb_batch, self.seq, hidden))
            shape_ok = self.seq % 8 == 0 and hidden % 64 == 0 and (self.mb_batch * self.seq) % 128 == 0
            if spans and spans[0].head is not None:
                shape_ok = shape_ok and attention_supported(
                    self.seq, spans[0].head.attention.self.attention_head_size)
            in_ok, out_ok = in_ok and shape_ok, out_ok and shape_ok
        if multi:
            flags: List[tuple] = [None] * dist.get_world_size(self.group)  # type: ignore[list-item]
            dist.all_gather_object(flags, (self.s, in_ok, out_ok, hidden), group=self.group)
            by_stage = {f[0]: f for f in flags}
            if not self.is_first:
                self.in_fused = want_fused and by_stage[self.s - 1][2] and in_ok
            if not self.is_last:
                self.out_fused = want_fused and by_stage[self.s + 1][1] and out_ok
            any_fused = any(
                by_stage[k][2] and by_stage[k + 1][1] for k in range(self.P - 1)) and want_fused
            if any_fused:
                # collective: every rank participates in the handle exchange
                from .p2p import FusedBoundaryManager

                hid = max(f[3] for f in flags)
                self.fused = FusedBoundaryManager(
                    self.s, self.P, self.stage_to_rank, self.m, self.mb_batch * self.seq, hid,
                    self.mb_batch * self.seq, self.device, group=self.group)
            if (not self.is_first and not self.in_fused) or (not self.is_last and not self.out_fused):
                from .comm import TorchDistComm

                self.comm = TorchDistComm(self.device, group=self.group)
        # only an optimizer whose step() is pure device work may be captured (a torch.optim class
        # behind TorchOptimizerAdapter keeps host-side state and refreshes the bf16 shadows through
        # a host-side version check: replaying it would train on stale weights)
        self.graphable = self._want_graph and self._native_active() and \
            (self.is_first or self.in_fused) and (self.is_last or self.out_fused) and \
            bool(getattr(self.optimizer, "graph_safe", False))
        if self.graphable:
            # device timers cannot be recorded inside a captured graph
            self.stage._record_forward_time = False
            self.stage._logger = None
        self._configure_wgrad(multi)
        self._order = (one_f_one_b_order if self.schedule == "1f1b" else sequential_order)(
            self.s, self.P, self.m)
        self._setup_done = True

    @staticmethod
    def _hidden_size(span) -> int:
        if span.head is not None:
            return span.head.attention.output.dense.weight.shape[0]
        if span.body is not None:
            return span.body.intermediate.dense_act.weight.shape[1]
        return span.tail.output.dense.weight.shape[0]

    # ------------------------------------------------------------------ per micro-batch work
    def _stage_inputs(self, j: int, chunks):
        if self.is_first:
            return tuple(c[j] for c in chunks)
        if self.in_fused:
            ch = self.fused.prev
            from ..ops import native as nat

            rows = self.mb_batch * self.seq
            # the additive mask rides next to the activation slot under its own flag
            nat.ext().wait_flags(ch.local.mask_flag_ptr(j), 1, ch.epoch_ptr, 1, ch.error_ptr,
                                 torch.cuda.current_stream().cuda_stream)
            x = ch.act_view(j, rows, ch.cols).view(self.mb_batch, self.seq, ch.cols)
            x.requires_grad_(True)
            mask = ch.mask_view(j, self.mb_batch * self.seq).view(self.mb_batch, 1, 1, self.seq)
            return (x, mask)
        return None  # filled by the comm path

    def _forward(self, j: int, args, labels_chunks):
        st = self.stage
        st.microbatch = j
        st.in_channel = self.fused.prev if self.in_fused else None
        st.out_channel = self.fused.next if self.out_fused else None
        if self.out_fused and not self.is_first:
            # the mask travels with the activation (own flag); relay it as early as possible
            self.fused.next.send_mask(args[-1], j)
        self._mark(("F", j, "begin"))
        outs = st(*args)
        self._mark(("F", j, "end"))
        if self.out_fused and self.is_first:
            self.fused.next.send_mask(outs[-1], j)  # produced by the embeddings of this stage
        loss = None
        if self.is_last:
            logits = outs[0]
            if hasattr(self.loss_fn, "fused") and logits.is_cuda and self._loss_acc.dtype == torch.float32:
                # (dlogits,) instead of a scalar loss: see _NativeCrossEntropy.fused
                loss = (self.loss_fn.fused(logits, labels_chunks[j], 1.0 / self.m,
                                           self._loss_acc.view(1)),)
            else:
                loss = self.loss_fn(logits, labels_chunks[j]) / self.m
                self._loss_acc += loss.detach().float()
        return outs, loss

    def _backward(self, j: int, outs, loss, grads, args):
        st = self.stage
        st.microbatch = j
        st.in_channel = self.fused.prev if self.in_fused else None
        st.out_channel = self.fused.next if self.out_fused else None
        # Weight gradients of the PREVIOUS micro-batch run now, i.e. in front of the kernel that
        # will wait for this micro-batch's incoming gradient: during the 1F1B cool-down they fill
        # what would otherwise be pipeline bubble, and they never delay the input gradient that
        # the previous stage is waiting for.
        self._flush_wgrads()
        self._mark(("B", j, "begin"))
        st.begin_backward()
        if self.is_last:
            if isinstance(loss, tuple):
                torch.autograd.backward([outs[0]], [loss[0].to(outs[0].dtype)])
            else:
                loss.backward()
        elif self.out_fused:
            dummy = outs[0]
            torch.autograd.backward([dummy], [torch.zeros_like(dummy)])
        else:
            ts, gs = [], []
            for o, g in zip(outs, grads):
                if g is not None and torch.is_tensor(o) and o.requires_grad:
                    ts.append(o)
                    gs.append(g.to(o.dtype))
            torch.autograd.backward(ts, gs)
        st.end_backward()
        self._mark(("B", j, "end"))
        if self.is_first or self.in_fused:
            return None
        return self._in_grads(args)

    def _slowdown_factor(self) -> float:
        return float(getattr(self.stage, "_slowdown", 0) or 0)

    # ------------------------------------------------------------------ comm helpers (unfused)
    @staticmethod
    def _diff_flags(tensors) -> List[bool]:
        """Which boundary tensors carry gradients: floating tensors, except a trailing additive
        mask when several tensors cross the boundary.  Both sides of a link apply this rule, so
        gradient messages need no metadata handshake."""
        n = len(tensors)
        return [torch.is_tensor(t) and t.is_floating_point() and (i < n - 1 or n == 1)
                for i, t in enumerate(tensors)]

    def _recv_forward(self):
        outs, reqs = self.comm.recv(self.prev_rank, "fwd")
        self.comm.wait(reqs)
        return self._prep_inputs(outs)

    def _prep_inputs(self, tensors):
        for t, d in zip(tensors, self._diff_flags(tensors)):
            if d:
                t.requires_grad_(True)
        return tuple(tensors)

    def _grad_metas(self, outs):
        return [(o.dtype, tuple(o.shape)) if d else None
                for o, d in zip(outs, self._diff_flags(outs))]

    def _in_grads(self, args):
        out = []
        for a, d in zip(args, self._diff_flags(args)):
            if not d:
                out.append(None)
            else:
                out.append(a.grad if a.grad is not None else torch.zeros_like(a))
        return out

    def _send_forward(self, outs):
        self._pending_sends += self.comm.send([o.detach() if torch.is_tensor(o) else None
                                               for o in outs], self.next_rank, "fwd")

    def _recv_backward(self, outs):
        grads, reqs = self.comm.recv(self.next_rank, "bwd", metas=self._grad_metas(outs))
        self.comm.wait(reqs)
        return grads

    def _send_backward(self, in_grads):
        self._pending_sends += self.comm.send(in_grads, self.prev_rank, "bwd", with_meta=False)

    def _send_forward_recv_backward(self, outs):
        g, reqs = self.comm.exchange([o.detach() if torch.is_tensor(o) else None for o in outs],
                                     self.next_rank, "fwd", self.next_rank, "bwd",
                                     recv_metas=self._grad_metas(outs), send_with_meta=True)
        self.comm.wait(reqs)
        return g

    def _send_backward_recv_forward(self, in_grads):
        metas = self.comm.cached_meta(self.prev_rank, "fwd")
        x, reqs = self.comm.exchange(in_grads, self.prev_rank, "bwd", self.prev_rank, "fwd",
                                     recv_metas=metas)
        self.comm.wait(reqs)
        return self._prep_inputs(x)

    # ------------------------------------------------------------------ one optimisation step
    def _step_body(self, inputs, labels):
        from ..models.bert_layers import advance_rng

        if self.fused is not None:
            self.fused.begin_step()
        if self._advance_rng and self._native_active():
            advance_rng()
        self._loss_acc.zero_()
        self._trace_tags = []
        self._mark(("STEP", 0, "begin"))
        chunks = [t.chunk(self.m, dim=0) for t in inputs] if self.is_first else None
        label_chunks = labels.chunk(self.m, dim=0) if (self.is_last and labels is not None) else None
        need_recv_f = not self.is_first and not self.in_fused
        need_send_f = not self.is_last and not self.out_fused
        need_recv_b = need_send_f
        need_send_b = need_recv_f
        saved = {}
        order = self._order
        pending_in = None       # input received together with a backward send
        pending_grad = None     # gradient received together with a forward send
        for idx, (kind, j) in enumerate(order):
            nxt = order[idx + 1] if idx + 1 < len(order) else None
            if kind == "F":
                if need_recv_f:
                    args = pending_in if pending_in is not None else self._recv_forward()
                    pending_in = None
                else:
                    args = self._stage_inputs(j, chunks)
                outs, loss = self._forward(j, args, label_chunks)
                saved[j] = (args, outs, loss)
                if need_send_f:
                    if nxt is not None and nxt[0] == "B":
                        pending_grad = self._send_forward_recv_backward(outs)
                    else:
                        self._send_forward(outs)
            else:
                args, outs, loss = saved.pop(j)
                grads = None
                if need_recv_b:
                    grads = pending_grad if pending_grad is not None else self._recv_backward(outs)
                    pending_grad = None
                in_grads = self._backward(j, outs, loss, grads, args)
                if need_send_b:
                    if nxt is not None and nxt[0] == "F":
                        pending_in = self._send_backward_recv_forward(in_grads)
                    else:
                        self._send_backward(in_grads)
        self._flush_wgrads()
        self._join_wgrads()
        if self.fused is not None:
            self.fused.end_of_backward()
        self._mark(("OPT", 0, "begin"))
        self.optimizer.step()
        self._mark(("OPT", 0, "end"))
        if self.comm is not None:
            self.comm.wait(self._pending_sends)
            self._pending_sends = []

    def train_step(self, inputs: Optional[Sequence[torch.Tensor]] = None,
                   labels: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """Run one optimisation step; returns the (mean) loss tensor on the last stage."""
        if not self._setup_done:
            self._setup(inputs)
            self._loss_acc = torch.zeros((), dtype=torch.float32, device=self.device)
        self._check_batch(inputs, labels)
        if not self.graphable:
            self._step_body(inputs, labels)
            return self._loss_acc if self.is_last else None
        # ---- CUDA-graph path: static input buffers, 3 eager steps, then capture + replay ----
        if self._static_inputs is None:
            self._static_inputs = [t.clone() for t in inputs] if self.is_first else []
            self._static_labels = labels.clone() if (self.is_last and labels is not None) else None
        if self.is_first:
            for s, t in zip(self._static_inputs, inputs):
                s.copy_(t, non_blocking=True)
        if self._static_labels is not None and labels is not None:
            self._static_labels.copy_(labels, non_blocking=True)
        if self._graph is None and self._eager_steps < 3:
            self._step_body(self._static_inputs, self._static_labels)
            self._eager_steps += 1
            return self._loss_acc if self.is_last else None
        if self._graph is None:
            torch.cuda.synchronize(self.device)
            from ..ops import native as nat

            g = torch.cuda.CUDAGraph()
            before = nat.launch_count()
            with torch.cuda.graph(g):
                self._step_body(self._static_inputs, self._static_labels)
            self.launches_per_step = nat.launch_count() - before
            self._graph = g
            # capture only records: replay right away so that this step's batch is trained on
            self._graph.replay()
            return self._loss_acc if self.is_last else None
        self._graph.replay()
        return self._loss_acc if self.is_last else None

    # ------------------------------------------------------------------ plain forward (eval)
    @torch.no_grad()
    def forward_only(self, inputs: Optional[Sequence[torch.Tensor]] = None):
        """Sequential forward through the pipeline without gradients (logits on the last stage)."""
        if self.P == 1:
            return self.stage(*inputs)
        from .comm import TorchDistComm

        comm = self.comm or TorchDistComm(self.device, group=self.group)
        if self.is_first:
            args = tuple(inputs)
        else:
            args, reqs = comm.recv(self.prev_rank, "eval")
            comm.wait(reqs)
        st = self.stage
        st.in_channel = st.out_channel = None
        outs = st(*args)
        if not self.is_last:
            comm.wait(comm.send(list(outs), self.next_rank, "eval"))
            return None
        return outs

    def close(self) -> None:
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)  # nothing of ours may still touch a peer region
        if self.fused is not None:
            self.fused.close()
            self.fused = None
        self._release_wgrad_switches()
