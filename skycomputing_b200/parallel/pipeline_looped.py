"""Looped ("breadth-first") pipeline engine: v virtual stages per rank.

A plain 1F1B step costs ``m x T + (P - 1) x (F + B)``: the fill / drain term is a whole stage's
forward + backward per pipeline hop and dominates at 8 GPUs (profiles/bench_history.md: 9.4 of
21.2 ms).  Here every rank owns v NON-adjacent chunks of the model (virtual stage k = chunk k // P
of rank k % P, ``Allocator.looped_allocate``), the ranks form a ring, and a micro-batch visits
every rank v times.  Each rank runs, per step,

    for c in chunks:            for j in micro-batches:  forward (c, j)
    for c in reversed(chunks):  for j in micro-batches:  backward(c, j)

(the breadth-first order of Lamy-Poirier, "Breadth-first pipeline parallelism", 2022).  A hop now
costs 1/v of a rank's work, so the step is ``m x T + (P - 1) x (F + B) / v`` as long as
``m >= P``; activation memory grows to all micro-batches of all chunks, which 180 GB of HBM absorb
easily for the models this framework targets.  Weight gradients use the same deferral as the
plain engine.

Transport: ``torch.distributed`` point-to-point by default (gloo on CPU, NCCL on GPUs) - both ends
of a link post their transfers in the same (chunk, micro-batch) order, so plain FIFO matching is
enough and no tags are needed.  ``boundary="fused"`` (``SKY_LOOPED_FUSED=1``) switches to the
plain engine's peer-memory boundary: the ranks form a RING of ``FusedChannel``s (incl. the
wrap-around link), one slot per (chunk, micro-batch), and the whole step is captured into one CUDA
graph.  The p2p path is covered by the CPU tests (tests/test_pipeline_cpu.py); the fused path is
written against the same kernels / flag protocol but has not been run on GPUs yet (DESIGN.md §7),
which is why it is opt-in.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import torch
import torch.distributed as dist

from ..ops.native import attention_supported
from .comm import TorchDistComm
from .engine_base import EngineBase


def looped_order(num_chunks: int, micro_batches: int) -> List[tuple]:
    """[('F' | 'B', chunk, micro_batch)] for one rank."""
    order = [("F", c, j) for c in range(num_chunks) for j in range(micro_batches)]
    order += [("B", c, j) for c in reversed(range(num_chunks)) for j in range(micro_batches)]
    return order


class LoopedPipelineEngine(EngineBase):
    def __init__(self, stages: Sequence, virtual_indices: Sequence[int], num_ranks: int,
                 ring: Sequence[int], device: torch.device, optimizer,
                 loss_fn: Optional[Callable] = None, micro_batches: int = 1, group=None,
                 advance_rng: bool = True, boundary: str = "dist", use_cuda_graph: bool = True):
        """``stages[i]`` is the ModuleWrapper of virtual stage ``virtual_indices[i]``; ``ring[p]`` is
        the process rank at ring position p (virtual stage k lives at position k % num_ranks)."""
        self.stages = list(stages)
        self.vidx = list(virtual_indices)
        self.P = num_ranks
        self.v = len(self.stages)
        self.total = self.P * self.v
        assert self.P >= 2, "a looped pipeline needs at least two ranks"
        assert self.vidx == sorted(self.vidx) and len(set(k % self.P for k in self.vidx)) == 1
        self.pos = self.vidx[0] % self.P
        self.s = self.pos                                 # ring position (trace / log naming)
        assert self.vidx == [c * self.P + self.pos for c in range(self.v)], self.vidx
        self.ring = list(ring)
        self.device = device
        self.optimizer = optimizer
        self.loss_fn = loss_fn
        self.m = micro_batches
        self.group = group
        self.prev_rank = self.ring[(self.pos - 1) % self.P]
        self.next_rank = self.ring[(self.pos + 1) % self.P]
        self.is_first = self.vidx[0] == 0                 # owns the stage that reads the data
        self.is_last = self.vidx[-1] == self.total - 1    # owns the stage that computes the loss
        self._comm: Optional[TorchDistComm] = None       # created on first use (p2p path only)
        self._loss_acc: Optional[torch.Tensor] = None
        self._advance_rng = advance_rng
        self._pending: list = []
        self._order = looped_order(self.v, self.m)
        for st in self.stages:
            st.engine_managed_backward = True
        # attributes the Runner / bench read on any engine
        self.schedule = "looped"
        self.fused = None
        self.in_fused = self.out_fused = False
        self.launches_per_step = 0
        self._graph = None
        self._init_common()
        self._setup_done = False
        self.boundary = boundary
        self._want_graph = use_cuda_graph and device.type == "cuda"
        self.graphable = False
        self._static_inputs: Optional[list] = None
        self._static_labels: Optional[torch.Tensor] = None
        self._eager_steps = 0
        self.mb_batch = self.seq = 0

    # ------------------------------------------------------------------ helpers
    @property
    def comm(self) -> TorchDistComm:
        if self._comm is None:
            self._comm = TorchDistComm(self.device, group=self.group)   # eval-only use
        return self._comm

    @staticmethod
    def _diff_flags(tensors) -> List[bool]:
        n = len(tensors)
        return [torch.is_tensor(t) and t.is_floating_point() and (i < n - 1 or n == 1)
                for i, t in enumerate(tensors)]

    def _prep_inputs(self, tensors):
        for t, d in zip(tensors, self._diff_flags(tensors)):
            if d:
                t.requires_grad_(True)
        return tuple(tensors)

    def _slowdown_factor(self) -> float:
        return max(float(getattr(st, "_slowdown", 0) or 0) for st in self.stages)

    def _trace_slots(self) -> int:
        return 8 * (2 * self.v * self.m + 4) + 64

    # ------------------------------------------------------------------ setup (collective)
    def _setup(self, inputs) -> None:
        self._loss_acc = torch.zeros((), dtype=torch.float32, device=self.device)
        self._configure_wgrad(True)
        want_fused = self.boundary in ("auto", "fused") and self._native_active()
        shape = [0, 0]
        if self.is_first:
            shape = [inputs[0].shape[0] // self.m, int(inputs[0].shape[1]) if inputs[0].dim() > 1 else 0]
        box = [shape]
        dist.broadcast_object_list(box, src=self.ring[0], group=self.group)
        self.mb_batch, self.seq = box[0]
        ok, hidden = False, 0
        if want_fused:
            ok = True
            for c, st in enumerate(self.stages):
                k = self.vidx[c]
                spans = st.spans()
                if spans:
                    sp = spans[0]
                    if sp.head is not None:
                        hidden = sp.head.attention.output.dense.weight.shape[0]
                        ok = ok and attention_supported(
                            self.seq, sp.head.attention.self.attention_head_size)
                in_ok, out_ok = st.fused_boundary_support((self.mb_batch, self.seq, hidden))
                ok = ok and (in_ok or k == 0) and (out_ok or k == self.total - 1)
            ok = ok and self.seq % 8 == 0 and hidden > 0 and hidden % 64 == 0 and \
                (self.mb_batch * self.seq) % 128 == 0
        flags = [None] * dist.get_world_size(self.group)
        dist.all_gather_object(flags, (bool(ok), int(hidden)), group=self.group)
        if want_fused and all(f[0] for f in flags):
            from .p2p import FusedBoundaryManager

            rows = self.mb_batch * self.seq
            self.fused = FusedBoundaryManager(self.pos, self.P, self.ring, self.v * self.m, rows,
                                              max(f[1] for f in flags), rows, self.device,
                                              group=self.group, ring=True)
            self.in_fused = self.out_fused = True
            self.graphable = self._want_graph and bool(getattr(self.optimizer, "graph_safe", False))
            if self.graphable:
                for st in self.stages:
                    st._record_forward_time = False
                    st._logger = None
        if self.fused is None:
            # collective: one communicator per direction so crossed sends cannot dead-lock NCCL
            self._comm = TorchDistComm(self.device, group=self.group, directional=True)
        self._setup_done = True

    def _fused_inputs(self, slot: int):
        from ..ops import native as nat

        ch = self.fused.prev
        rows = self.mb_batch * self.seq
        nat.ext().wait_flags(ch.local.mask_flag_ptr(slot), 1, ch.epoch_ptr, 1, ch.error_ptr,
                             torch.cuda.current_stream().cuda_stream)
        x = ch.act_view(slot, rows, ch.cols).view(self.mb_batch, self.seq, ch.cols)
        x.requires_grad_(True)
        mask = ch.mask_view(slot, rows).view(self.mb_batch, 1, 1, self.seq)
        return (x, mask)

    def _step_body_fused(self, inputs, labels) -> None:
        """The same (chunk, micro-batch) order with every boundary in peer memory: no host-side
        transfers at all, the kernels of neighbouring ranks hand panels to each other."""
        from ..models.bert_layers import advance_rng

        self.fused.begin_step()
        if self._advance_rng:
            advance_rng()
        self._loss_acc.zero_()
        self._trace_tags = []
        self._mark(("STEP", 0, "begin"))
        chunks_in = [t.chunk(self.m, dim=0) for t in inputs] if self.is_first else None
        label_chunks = labels.chunk(self.m, dim=0) if (self.is_last and labels is not None) else None
        saved = {}
        for kind, c, j in self._order:
            k = self.vidx[c]
            st = self.stages[c]
            # a link's slots are numbered by the CONSUMER's chunk: inbound = this chunk, outbound =
            # the chunk of virtual stage k + 1 (the same number except on the wrap-around link
            # from the last ring position to the first, where it is c + 1)
            slot = c * self.m + j
            out_slot = ((k + 1) // self.P) * self.m + j
            first_stage, last_stage = k == 0, k == self.total - 1
            st.microbatch = (slot, out_slot)
            st.in_channel = None if first_stage else self.fused.prev
            st.out_channel = None if last_stage else self.fused.next
            if kind == "F":
                args = tuple(t[j] for t in chunks_in) if first_stage else self._fused_inputs(slot)
                if not last_stage and not first_stage:
                    self.fused.next.send_mask(args[-1], out_slot)   # the mask travels with the slot
                self._mark(("F", slot, "begin"))
                outs = st(*args)
                self._mark(("F", slot, "end"))
                if not last_stage and first_stage:
                    self.fused.next.send_mask(outs[-1], out_slot)   # produced by the embeddings here
                loss = None
                if last_stage:
                    if hasattr(self.loss_fn, "fused"):
                        loss = (self.loss_fn.fused(outs[0], label_chunks[j], 1.0 / self.m,
                                                   self._loss_acc.view(1)),)
                    else:
                        loss = self.loss_fn(outs[0], label_chunks[j]) / self.m
                        self._loss_acc += loss.detach().float()
                saved[(c, j)] = (outs, loss)
            else:
                outs, loss = saved.pop((c, j))
                self._flush_wgrads()
                self._mark(("B", slot, "begin"))
                st.begin_backward()
                if last_stage:
                    if isinstance(loss, tuple):
                        torch.autograd.backward([outs[0]], [loss[0].to(outs[0].dtype)])
                    else:
                        loss.backward()
                else:
                    torch.autograd.backward([outs[0]], [torch.zeros_like(outs[0])])
                st.end_backward()
                self._mark(("B", slot, "end"))
        self._flush_wgrads()
        self._join_wgrads()
        self.fused.end_of_backward()
        self._mark(("OPT", 0, "begin"))
        self.optimizer.step()
        self._mark(("OPT", 0, "end"))

    # ------------------------------------------------------------------ one optimisation step
    def train_step(self, inputs: Optional[Sequence[torch.Tensor]] = None,
                   labels: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        if not self._setup_done:
            self._setup(inputs)
        self._check_batch(inputs, labels)
        if self.fused is not None:
            return self._train_step_fused(inputs, labels)
        if self._advance_rng and self._native_active():
            from ..models.bert_layers import advance_rng

            advance_rng()
        self._loss_acc.zero_()
        chunks_in = [t.chunk(self.m, dim=0) for t in inputs] if self.is_first else None
        label_chunks = labels.chunk(self.m, dim=0) if (self.is_last and labels is not None) else None
        saved = {}
        for kind, c, j in self._order:
            k = self.vidx[c]
            st = self.stages[c]
            st.microbatch = c * self.m + j
            st.in_channel = st.out_channel = None
            first_stage, last_stage = k == 0, k == self.total - 1
            if kind == "F":
                if first_stage:
                    args = tuple(t[j] for t in chunks_in)
                else:
                    got, reqs = self.comm.recv(self.prev_rank, f"fwd{c}")
                    self.comm.wait(reqs)
                    args = self._prep_inputs(got)
                outs = st(*args)
                loss = None
                if last_stage:
                    loss = self.loss_fn(outs[0], label_chunks[j]) / self.m
                    self._loss_acc += loss.detach().float()
                else:
                    self._pending += self.comm.send(
                        [o.detach() if torch.is_tensor(o) else None for o in outs],
                        self.next_rank, f"fwd{c}")
                saved[(c, j)] = (args, outs, loss)
            else:
                args, outs, loss = saved.pop((c, j))
                self._flush_wgrads()
                st.begin_backward()
                if last_stage:
                    loss.backward()
                else:
                    metas = [(o.dtype, tuple(o.shape)) if d else None
                             for o, d in zip(outs, self._diff_flags(outs))]
                    grads, reqs = self.comm.recv(self.next_rank, f"bwd{c}", metas=metas)
                    self.comm.wait(reqs)
                    ts, gs = [], []
                    for o, g in zip(outs, grads):
                        if g is not None and torch.is_tensor(o) and o.requires_grad:
                            ts.append(o)
                            gs.append(g.to(o.dtype))
                    torch.autograd.backward(ts, gs)
                st.end_backward()
                if not first_stage:
                    in_grads = [(a.grad if a.grad is not None else torch.zeros_like(a)) if d else None
                                for a, d in zip(args, self._diff_flags(args))]
                    self._pending += self.comm.send(in_grads, self.prev_rank, f"bwd{c}",
                                                    with_meta=False)
        self._flush_wgrads()
        self._join_wgrads()
        self.optimizer.step()
        self.comm.wait(self._pending)
        self._pending = []
        return self._loss_acc if self.is_last else None

    def _train_step_fused(self, inputs, labels):
        """Static buffers, 3 eager steps, then one CUDA graph per step (as in PipelineEngine)."""
        out = self._loss_acc if self.is_last else None
        if not self.graphable:
            self._step_body_fused(inputs, labels)
            return out
        if self._static_inputs is None:
            self._static_inputs = [t.clone() for t in inputs] if self.is_first else []
            self._static_labels = labels.clone() if (self.is_last and labels is not None) else None
        if self.is_first:
            for s_, t in zip(self._static_inputs, inputs):
                s_.copy_(t, non_blocking=True)
        if self._static_labels is not None and labels is not None:
            self._static_labels.copy_(labels, non_blocking=True)
        if self._graph is None and self._eager_steps < 3:
            self._step_body_fused(self._static_inputs, self._static_labels)
            self._eager_steps += 1
            return out
        if self._graph is None:
            from ..ops import native as nat

            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            before = nat.launch_count()
            with torch.cuda.graph(g):
                self._step_body_fused(self._static_inputs, self._static_labels)
            self.launches_per_step = nat.launch_count() - before
            self._graph = g
        self._graph.replay()
        return out

    # ------------------------------------------------------------------ plain forward (eval)
    @torch.no_grad()
    def forward_only(self, inputs: Optional[Sequence[torch.Tensor]] = None):
        outs = None
        for c, st in enumerate(self.stages):
            k = self.vidx[c]
            if k == 0:
                args = tuple(inputs)
            else:
                args, reqs = self.comm.recv(self.prev_rank, f"eval{c}")
                self.comm.wait(reqs)
            st.in_channel = st.out_channel = None
            outs = st(*args)
            if k != self.total - 1:
                self.comm.wait(self.comm.send(list(outs), self.next_rank, f"eval{c}"))
                outs = None
        return outs

    def close(self) -> None:
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)
        if self.fused is not None:
            self.fused.close()
            self.fused = None
        self._release_wgrad_switches()

    @staticmethod
    def barrier(group=None) -> None:
        if dist.is_available() and dist.is_initialized():
            dist.barrier(group=group)
