"""BERT layer library, split into the reference's allocatable units.

Registered names and calling conventions are those of scaelum/model/bert_layers.py:171-395:

    BertEmbeddings(config)            (input_ids, token_type_ids, attention_mask) -> (emb, ext_mask)
    BertLayer_Head(config)            (hidden, mask)            -> (attn_out, mask)
    BertLayer_Body(config)            (attn_out, mask)          -> (inter, attn_out, mask)
    BertLayer_Tail(config)            (inter, attn_out, mask)   -> (hidden, mask)
    BertPooler(config)                (hidden, mask)            -> pooled
    BertTailForClassification(hidden_dropout_prob, hidden_size, num_classes)   pooled -> logits

Parameter names match the reference (``attention.self.query.weight`` ...), so layer-indexed
checkpoints interchange.  Every layer has two execution paths behind the same class:

* ``torch``  - fp32 eager PyTorch with exactly the reference's math.  It is the numerics oracle for
  the kernel tests and the CPU path (BASELINE config 1 runs on it over gloo).
* ``native`` - bf16 sm_100a kernels (tcgen05 GEMMs / attention, fused LayerNorm, in-kernel
  dropout) through ``skycomputing_b200.ops.functions``.  Consecutive Head/Body/Tail layers of one
  block are executed as ONE autograd node (``BertSpan``); the stage runtime builds those spans.

``set_backend("auto" | "torch" | "native")`` selects the path; ``auto`` means native whenever the
input lives on a CUDA device and the extension is built.
"""
from __future__ import annotations

import math
from typing import List

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..registry import LAYER
from .bert import BertConfig

_BACKEND = "auto"


def set_backend(name: str) -> None:
    global _BACKEND
    assert name in ("auto", "torch", "native"), name
    _BACKEND = name


def get_backend() -> str:
    return _BACKEND


def _nat():
    from ..ops import native

    return native


def _native_enabled(t: torch.Tensor) -> bool:
    if _BACKEND == "torch" or not t.is_cuda:
        if _BACKEND == "native" and not t.is_cuda:
            raise RuntimeError("backend 'native' requires CUDA tensors")
        return False
    nat = _nat()
    if nat.available():
        return True
    if _BACKEND == "native":
        nat.ext()  # raises with the build hint
    raise RuntimeError(
        "CUDA tensors reached a skycomputing_b200 layer but the sm_100a extension is not built; "
        "run __graft_entry__.build() (or set_backend('torch') to use the eager oracle on purpose)"
    )


# device-resident dropout RNG shared by all native layers of this process
_RNG = {}
_RNG_STREAM_COUNTER = [0]


def default_rng(device: torch.device):
    key = (device.type, device.index)
    if key not in _RNG:
        _RNG[key] = _nat().RngState(torch.initial_seed(), device=device)
    return _RNG[key]


def advance_rng(inc: int = 1) -> None:
    """Advance the dropout step counter (one launch per device; CUDA-graph capturable)."""
    for r in _RNG.values():
        r.advance(inc)


def _next_rng_base() -> int:
    _RNG_STREAM_COUNTER[0] += 8
    return _RNG_STREAM_COUNTER[0]


# --------------------------------------------------------------------------------------------
# activations (reference: bert_layers.py:21-57)
# --------------------------------------------------------------------------------------------
def gelu(x):
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def bias_gelu(bias, y):
    return gelu(bias + y)


def bias_gelu_training(bias, y):
    """Training-time variant of bias_gelu (scaelum bert_layers.py:36-38): bias add + library erf-GELU."""
    return torch.nn.functional.gelu(bias + y)


def bias_tanh(bias, y):
    return torch.tanh(bias + y)


def swish(x):
    return x * torch.sigmoid(x)


ACT2FN = {"gelu": gelu, "bias_gelu": bias_gelu, "bias_tanh": bias_tanh, "relu": F.relu,
          "swish": swish, "tanh": torch.tanh}


class LinearActivation(nn.Module):
    """Linear whose bias is folded into the activation (reference: bert_layers.py:60-108)."""

    def __init__(self, in_features: int, out_features: int, act="gelu", bias: bool = True):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        self.act_name = act if isinstance(act, str) else None
        # reference semantics (bert_layers.py:73-84): with a bias, "gelu" means "bias_gelu" - the
        # bias is handed to the activation instead of to F.linear; "bias_*" names are accepted
        # directly.  `act_fn` is the plain activation, `biased_act_fn(bias, y)` the folded form.
        self.biased_act_fn = None
        if isinstance(act, str):
            base = act[5:] if act.startswith("bias_") else act
            folded = "bias_" + base
            if folded in ACT2FN:
                self.biased_act_fn = ACT2FN[folded]
            if base in ACT2FN:
                self.act_fn = ACT2FN[base]
            elif self.biased_act_fn is not None:
                fn = self.biased_act_fn
                self.act_fn = lambda y: fn(torch.zeros((), dtype=y.dtype, device=y.device), y)
            else:
                raise KeyError(f"unknown activation {act!r}; known: {sorted(ACT2FN)}")
        else:
            self.act_fn = act
        self.weight = nn.Parameter(torch.empty(out_features, in_features))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_features))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self) -> None:
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            bound = 1 / math.sqrt(self.in_features)
            nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, x):
        y = F.linear(x, self.weight, None)
        if self.bias is None:
            return self.act_fn(y)
        if self.biased_act_fn is not None:
            return self.biased_act_fn(self.bias, y)
        return self.act_fn(y + self.bias)

    def extra_repr(self) -> str:
        return f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}"


class BertLayerNorm(nn.Module):
    """TF-style LayerNorm (epsilon inside the sqrt), reference: bert_layers.py:143-168."""

    def __init__(self, hidden_size: int, eps: float = 1e-12):
        super().__init__()
        self.shape = torch.Size((hidden_size,))
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(hidden_size))
        self.bias = nn.Parameter(torch.zeros(hidden_size))

    def forward(self, x):
        u = x.mean(-1, keepdim=True)
        s = (x - u).pow(2).mean(-1, keepdim=True)
        x = (x - u) / torch.sqrt(s + self.eps)
        return self.weight * x + self.bias


BertNonFusedLayerNorm = BertLayerNorm


# --------------------------------------------------------------------------------------------
# embeddings
# --------------------------------------------------------------------------------------------
@LAYER.register_module
class BertEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        config = BertConfig.from_dict(config) if isinstance(config, dict) else config
        self.word_embeddings = nn.Embedding(config.vocab_size, config.hidden_size)
        self.position_embeddings = nn.Embedding(config.max_position_embeddings, config.hidden_size)
        self.token_type_embeddings = nn.Embedding(config.type_vocab_size, config.hidden_size)
        self.LayerNorm = BertLayerNorm(config.hidden_size, eps=1e-12)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)
        self._native = None

    def _native_params(self):
        from ..ops.functions import EmbeddingParams

        if self._native is None:
            object.__setattr__(self, "_native", EmbeddingParams(self))
            self._native.rng_base = _next_rng_base()
        self._native.rng = default_rng(self.word_embeddings.weight.device)
        return self._native

    def forward(self, input_ids, token_type_ids, attention_mask):
        if _native_enabled(input_ids) and self.word_embeddings.weight.shape[1] % 4 == 0:
            from ..ops.functions import EmbeddingsFn

            ep = self._native_params()
            return EmbeddingsFn.apply(ep, self.training, None, 0, input_ids, token_type_ids,
                                      attention_mask, *ep.all_params())
        ext = attention_mask.unsqueeze(1).unsqueeze(2).to(dtype=self.word_embeddings.weight.dtype)
        ext = (1.0 - ext) * -10000.0
        seq_length = input_ids.size(1)
        position_ids = torch.arange(seq_length, dtype=torch.long, device=input_ids.device)
        position_ids = position_ids.unsqueeze(0).expand_as(input_ids)
        emb = (self.word_embeddings(input_ids) + self.position_embeddings(position_ids)
               + self.token_type_embeddings(token_type_ids))
        emb = self.dropout(self.LayerNorm(emb))
        return emb, ext


# --------------------------------------------------------------------------------------------
# transformer block pieces (oracle sub-modules keep the reference's attribute names)
# --------------------------------------------------------------------------------------------
class BertSelfAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        if config.hidden_size % config.num_attention_heads != 0:
            raise ValueError(
                "The hidden size (%d) is not a multiple of the number of attention heads (%d)"
                % (config.hidden_size, config.num_attention_heads))
        self.num_attention_heads = config.num_attention_heads
        self.attention_head_size = config.hidden_size // config.num_attention_heads
        self.all_head_size = self.num_attention_heads * self.attention_head_size
        self.query = nn.Linear(config.hidden_size, self.all_head_size)
        self.key = nn.Linear(config.hidden_size, self.all_head_size)
        self.value = nn.Linear(config.hidden_size, self.all_head_size)
        self.dropout = nn.Dropout(config.attention_probs_dropout_prob)

    def _split(self, x):
        return x.reshape(x.size()[:-1] + (self.num_attention_heads, self.attention_head_size)
                         ).permute(0, 2, 1, 3)

    def forward(self, hidden_states, attention_mask):
        q = self._split(self.query(hidden_states))
        k = self._split(self.key(hidden_states))
        v = self._split(self.value(hidden_states))
        scores = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(self.attention_head_size)
        scores = scores + attention_mask
        probs = self.dropout(F.softmax(scores, dim=-1))
        ctx = torch.matmul(probs, v).permute(0, 2, 1, 3).contiguous()
        return ctx.reshape(ctx.size()[:-2] + (self.all_head_size,))


class BertSelfOutput(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.LayerNorm = BertLayerNorm(config.hidden_size, eps=1e-12)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_states, input_tensor):
        return self.LayerNorm(self.dropout(self.dense(hidden_states)) + input_tensor)


class BertAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.self = BertSelfAttention(config)
        self.output = BertSelfOutput(config)

    def forward(self, input_tensor, attention_mask):
        return self.output(self.self(input_tensor, attention_mask), input_tensor)


class BertIntermediate(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense_act = LinearActivation(config.hidden_size, config.intermediate_size,
                                          act=config.hidden_act)

    def forward(self, hidden_states):
        return self.dense_act(hidden_states)


class BertOutput(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.intermediate_size, config.hidden_size)
        self.LayerNorm = BertLayerNorm(config.hidden_size, eps=1e-12)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_states, input_tensor):
        return self.LayerNorm(self.dropout(self.dense(hidden_states)) + input_tensor)


class BertSpan:
    """A contiguous run of Head/Body/Tail layers of ONE block executed as a single autograd node.

    Not an ``nn.Module`` (the layers stay owned by the stage's Sequential); the stage runtime
    creates spans from adjacent layers, a lone layer creates a one-element span for itself.
    """

    def __init__(self, head=None, body=None, tail=None):
        from ..ops.functions import SpanParams

        self.head, self.body, self.tail = head, body, tail
        self.params = SpanParams(head, body, tail)
        self.params.rng_base = _next_rng_base()
        self.in_channel = None   # parallel.p2p.FusedChannel feeding this span (stage input)
        self.out_channel = None  # channel this span's LayerNorm writes into (stage output)
        self.microbatch = 0

    @property
    def layers(self) -> List[nn.Module]:
        return [m for m in (self.head, self.body, self.tail) if m is not None]

    def supports(self, hidden: torch.Tensor) -> bool:
        H = hidden.shape[-1]
        if hidden.dim() != 3 or H % 8 != 0:
            return False
        if self.head is not None:
            # tcgen05 attention: head sizes 8..128 in steps of 8, any sequence length that is a
            # multiple of 8 (S = 128 / head size 64: single-tile kernels, else flash-style tiles)
            from ..ops.native import attention_supported

            if not attention_supported(hidden.shape[1], self.head.attention.self.attention_head_size):
                return False
        if self.body is not None and self.body.intermediate.dense_act.act_name not in ("gelu", "bias_gelu"):
            return False
        return True

    def __call__(self, *inputs):
        from ..ops.functions import BertSpanFn

        sp = self.params
        first = (self.head or self.body or self.tail)
        training = first.training
        dev = inputs[0].device
        sp.rng = default_rng(dev)
        inputs = tuple(t.to(torch.bfloat16) if (torch.is_tensor(t) and t.is_floating_point()
                                                and t.dim() == 3 and t.dtype != torch.bfloat16)
                       else t for t in inputs)
        out = BertSpanFn.apply(sp, training, self.in_channel, self.out_channel, self.microbatch,
                               len(inputs), *inputs, *sp.all_params())
        mask = inputs[-1]
        if self.tail is not None:
            return out, mask
        if self.body is not None:
            if self.head is not None:
                inter, attn_out = out
            else:
                inter, attn_out = out, inputs[0]
            return inter, attn_out, mask
        return out, mask


def _lone_span(layer, **kw) -> BertSpan:
    span = layer.__dict__.get("_lone_span")
    if span is None:
        span = BertSpan(**kw)
        object.__setattr__(layer, "_lone_span", span)
    return span


@LAYER.register_module
class BertLayer_Head(nn.Module):
    def __init__(self, config):
        super().__init__()
        config = BertConfig.from_dict(config) if isinstance(config, dict) else config
        self.attention = BertAttention(config)

    def forward(self, hidden_states, attention_mask):
        if _native_enabled(hidden_states):
            span = _lone_span(self, head=self)
            if span.supports(hidden_states):
                return span(hidden_states, attention_mask)
        hidden_states = hidden_states.float()
        return self.attention(hidden_states, attention_mask), attention_mask


@LAYER.register_module
class BertLayer_Body(nn.Module):
    def __init__(self, config):
        super().__init__()
        config = BertConfig.from_dict(config) if isinstance(config, dict) else config
        self.intermediate = BertIntermediate(config)

    def forward(self, attention_output, attention_mask):
        if _native_enabled(attention_output):
            span = _lone_span(self, body=self)
            if span.supports(attention_output):
                return span(attention_output, attention_mask)
        attention_output = attention_output.float()
        return self.intermediate(attention_output), attention_output, attention_mask


@LAYER.register_module
class BertLayer_Tail(nn.Module):
    def __init__(self, config):
        super().__init__()
        config = BertConfig.from_dict(config) if isinstance(config, dict) else config
        self.output = BertOutput(config)

    def forward(self, intermediate_output, attention_output, attention_mask):
        if _native_enabled(attention_output):
            span = _lone_span(self, tail=self)
            if span.supports(attention_output):
                return span(intermediate_output, attention_output, attention_mask)
        out = self.output(intermediate_output.float(), attention_output.float())
        return out, attention_mask


@LAYER.register_module
class BertPooler(nn.Module):
    def __init__(self, config):
        super().__init__()
        config = BertConfig.from_dict(config) if isinstance(config, dict) else config
        self.dense_act = LinearActivation(config.hidden_size, config.hidden_size, act="tanh")
        self._native = None

    def _native_params(self):
        from ..ops.functions import SmallLinearParams

        if self._native is None:
            object.__setattr__(self, "_native", SmallLinearParams(
                self.dense_act.weight, self.dense_act.bias, act_tanh=True, first_token=True))
        return self._native

    def forward(self, hidden_states, attention_mask):
        if _native_enabled(hidden_states) and hidden_states.dim() == 3:
            from ..ops.functions import PoolerFn, SmallLinearFn

            lp = self._native_params()
            B, _S, H = hidden_states.shape
            if B % 8 == 0 and H % 8 == 0 and hidden_states.dtype == torch.bfloat16:
                return PoolerFn.apply(lp, hidden_states, *lp.all_params())  # tcgen05 GEMM path
            return SmallLinearFn.apply(lp, self.training, hidden_states, *lp.all_params())
        first_token_tensor = hidden_states[:, 0].float()
        return self.dense_act(first_token_tensor)


@LAYER.register_module
class BertTailForClassification(nn.Module):
    def __init__(self, hidden_dropout_prob, hidden_size, num_classes):
        super().__init__()
        self.num_classes = num_classes
        self.dropout = nn.Dropout(hidden_dropout_prob)
        self.classifier = nn.Linear(hidden_size, num_classes)
        self._native = None

    def _native_params(self):
        from ..ops.functions import SmallLinearParams

        if self._native is None:
            object.__setattr__(self, "_native", SmallLinearParams(
                self.classifier.weight, self.classifier.bias, act_tanh=False,
                first_token=False, p_drop=float(self.dropout.p)))
            self._native.rng_base = _next_rng_base()
        return self._native

    def forward(self, logits):
        if _native_enabled(logits) and logits.dim() == 2:
            from ..ops.functions import SmallLinearFn

            lp = self._native_params()
            lp.rng = default_rng(logits.device)
            return SmallLinearFn.apply(lp, self.training, logits, *lp.all_params()).view(
                -1, self.num_classes)
        logits = self.classifier(self.dropout(logits.float()))
        return logits.view(-1, self.num_classes)


def native_param_banks(module: nn.Module):
    """All ParamBanks of `module`'s native layers (created eagerly; used by the fused optimizer).

    For a stage (``ModuleWrapper``) the banks of its fused spans are returned, so that the
    optimizer and the forward pass share the same flat fp32 / bf16 buffers.
    """
    banks = []
    covered = set()
    # every stage runtime (ModuleWrapper) below `module` - `module` itself, or the chunks of a
    # looped pipeline held in a ModuleList - contributes the banks of ITS fused spans: building
    # lone per-layer spans for them instead would give the optimizer different flat buffers than
    # the ones the forward pass reads
    for m in module.modules():
        spans = getattr(m, "spans", None)
        if callable(spans):
            for span in spans():
                banks.extend(span.params.banks)
                covered.update(id(l) for l in span.layers)
    for m in module.modules():
        if id(m) in covered:
            continue
        if isinstance(m, BertEmbeddings):
            banks.extend(m._native_params().banks)
        elif isinstance(m, BertPooler):
            banks.extend(m._native_params().banks)
        elif isinstance(m, BertTailForClassification):
            banks.extend(m._native_params().banks)
        elif isinstance(m, BertLayer_Head):
            banks.extend(_lone_span(m, head=m).params.banks)
        elif isinstance(m, BertLayer_Body):
            banks.extend(_lone_span(m, body=m).params.banks)
        elif isinstance(m, BertLayer_Tail):
            banks.extend(_lone_span(m, tail=m).params.banks)
    return banks
