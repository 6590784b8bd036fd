"""The reference's OWN layer classes (the unmodified ``scaelum`` package) as the numerics oracle
(SURVEY §4: "each kernel vs the reference layer class with identical weights").  What the reference
computed is stored in tests/golden/reference_oracle_*.npz, so the suite runs without it:

* CPU: our state dicts have the reference's keys, shapes and order, and our fp32 eager path
  reproduces the reference's forward and backward to fp32 round-off for every registered BERT layer;
* GPU: the native sm_100a path at BERT-large geometry (H=1024, I=4096, 16 heads, 32 x 128 tokens)
  against scaelum/model/bert_layers.py:171-395 run in fp32, per-tensor relative L2 tolerances; and
  with dropout ON, against the reference classes fed the EXACT masks the kernels use (regenerated
  on the host from the dropout RNG state, which the test pins to the value the golden data used).

Weights and inputs come from seeded numpy generators, identical here and when the golden data was
made.  Every compared tensor is stored as a fixed sample of its nonzero elements (indices and
values) plus the L2 norm of the whole tensor.  To regenerate the golden data from an installed
copy of the reference (see baseline/README.md):

    python -m tests.test_reference_oracle --reference baseline/_ref
"""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

BLOCK = ["BertLayer_Head", "BertLayer_Body", "BertLayer_Tail"]
CPU_LAYERS = ["BertEmbeddings"] + BLOCK + ["BertPooler", "BertTailForClassification"]
# dropout RNG state {seed, step} and span stream base the dropout case pins for the native kernels
DROPOUT_SEED, DROPOUT_STEP, DROPOUT_BASE = 0x5EED, 1, 8


def _golden(name):
    with np.load(os.path.join(GOLDEN, f"reference_oracle_{name}.npz")) as z:
        return dict(z)


def _configs(hidden, heads, inter, p=0.0, vocab=1000):
    import skycomputing_b200 as sky  # noqa: F401
    from skycomputing_b200.models import BertConfig

    c = BertConfig(vocab, hidden_size=hidden, num_hidden_layers=1, num_attention_heads=heads,
                   intermediate_size=inter, max_position_embeddings=128,
                   hidden_dropout_prob=p, attention_probs_dropout_prob=p)
    return c


def _layer_kwargs(name, cfg):
    if name == "BertTailForClassification":
        return dict(hidden_dropout_prob=cfg.hidden_dropout_prob, hidden_size=cfg.hidden_size,
                    num_classes=3)
    return dict(config=dict(cfg.__dict__))


def _state_entries(layers):
    """'<layer index>|<key>|<shape>' for every state-dict entry, in state-dict order."""
    return [f"{i}|{k}|{','.join(map(str, v.shape))}"
            for i, l in enumerate(layers) for k, v in l.state_dict().items()]


def _load_seeded_weights(layers, entries, seed, std):
    """Loads N(0, std) into every entry (1 + N(0, std) for LayerNorm weights), drawn in the order of
    ``entries``; strict loading checks that the layers have exactly these keys."""
    rs = np.random.RandomState(seed)
    sds = [{} for _ in layers]
    for e in entries:
        i, key, shape = str(e).split("|")
        w = rs.standard_normal(tuple(int(s) for s in shape.split(","))) * std
        if key.endswith("LayerNorm.weight"):
            w += 1.0
        sds[int(i)][key] = torch.from_numpy(w.astype(np.float32))
    for l, sd in zip(layers, sds):
        l.load_state_dict(sd)


def _build_ours(names, cfg, device):
    import skycomputing_b200 as sky

    return [sky.build_layer(n, **_layer_kwargs(n, cfg)).to(device) for n in names]


def _chain(layers, inputs):
    x = inputs
    for l in layers:
        x = l(*x) if isinstance(x, (tuple, list)) else l(x)
    return x if isinstance(x, (tuple, list)) else (x,)


def _rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _vs_golden(golden, name, t):
    """(our sample, reference sample, our full-tensor norm, reference full-tensor norm)."""
    flat = t.detach().double().reshape(-1).cpu()
    idx = torch.from_numpy(golden[name + ".idx"].astype(np.int64))
    ref = torch.from_numpy(golden[name + ".val"]).double()
    return flat[idx], ref, float(flat.norm()), float(golden[name + ".norm"])


def _cpu_inputs(B=3, S=16, vocab=1000):
    rs = np.random.RandomState(3)
    ids = torch.from_numpy(rs.randint(0, vocab, (B, S)))
    tt = torch.from_numpy(rs.randint(0, 2, (B, S)))
    am = torch.ones(B, S, dtype=torch.long)
    am[1, 10:] = 0
    cot = torch.from_numpy(rs.standard_normal((B, 3)).astype(np.float32))
    return ids, tt, am, cot


def test_state_dicts_interchange_and_eager_path_equals_reference_cpu():
    from skycomputing_b200.models import set_backend

    golden = _golden("cpu")
    cfg = _configs(64, 4, 128)
    ours = _build_ours(CPU_LAYERS, cfg, "cpu")
    assert _state_entries(ours) == list(golden["state"])     # same keys, shapes and order
    _load_seeded_weights(ours, golden["state"], seed=10, std=0.1)
    ids, tt, am, cot = _cpu_inputs()
    set_backend("torch")
    try:
        out = _chain(ours, (ids, tt, am))[0]
        out.backward(cot)
    finally:
        set_backend("auto")
    o, r, on, rn = _vs_golden(golden, "out", out)
    torch.testing.assert_close(o, r, rtol=1e-5, atol=1e-6)
    assert on == pytest.approx(rn, rel=1e-5)
    for i, layer in enumerate(ours):
        for n, p in layer.named_parameters():
            o, r, on, rn = _vs_golden(golden, f"grad.{i}.{n}", p.grad)
            torch.testing.assert_close(o, r, rtol=1e-4, atol=1e-6, msg=n)
            assert on == pytest.approx(rn, rel=1e-4, abs=1e-6), n


def _block_inputs(B, S, H, seed=1):
    rs = np.random.RandomState(seed)
    x = torch.from_numpy(rs.standard_normal((B, S, H)).astype(np.float32))
    cot = torch.from_numpy(rs.standard_normal((B, S, H)).astype(np.float32))
    m = torch.ones(B, S)
    m[0, S - 30:] = 0
    m[B - 1, S // 2:] = 0
    ext = ((1.0 - m) * -10000.0).view(B, 1, 1, S)
    return x, ext, cot


def _native_stage(ours_layers):
    from skycomputing_b200.builder import ModuleWrapper, SequentialWrapper

    return ModuleWrapper(rank=0, module=SequentialWrapper(*ours_layers), module_to_cuda=True,
                         cuda_device=0)


def _check_block_against_golden(golden, layers, out, x_grad):
    """bf16 operands / fp32 accumulation vs the fp32 oracle: relative L2 error per tensor, on the
    stored sample and on the norm of the whole tensor."""
    for name, t, tol in (("out", out, 1.5e-2), ("x.grad", x_grad, 2.5e-2)):
        o, r, on, rn = _vs_golden(golden, name, t)
        assert _rel_l2(o, r) < tol, (name, _rel_l2(o, r))
        assert abs(on - rn) < tol * rn, (name, on, rn)
    worst = {}
    for i, layer in enumerate(layers):
        for n, p in layer.named_parameters():
            if n.endswith("key.bias"):
                _check_zero_gradient(layer, p)
                continue
            o, r, on, rn = _vs_golden(golden, f"grad.{i}.{n}", p.grad)
            worst[n] = max(worst.get(n, 0.0), _rel_l2(o, r), abs(on - rn) / rn)
    bad = {n: e for n, e in worst.items() if e > 3e-2}
    assert not bad, bad


@pytest.mark.gpu
def test_native_block_matches_reference_classes_at_bert_large_geometry():
    """H=1024, I=4096, 16 heads, 32 x 128 tokens (the benchmark's shapes: the GEMM + LayerNorm
    epilogue kernel, 256-wide tiles, 4-CTA clusters are what runs here), two blocks."""
    from skycomputing_b200.models import set_backend

    golden = _golden("block")
    torch.manual_seed(0)
    cfg = _configs(1024, 16, 4096, vocab=30522)
    ours = _build_ours(BLOCK * 2, cfg, "cuda")
    assert _state_entries(ours) == list(golden["state"])
    _load_seeded_weights(ours, golden["state"], seed=11, std=0.02)   # BERT-like scale
    B, S, H = 32, 128, 1024
    x, ext, cot = _block_inputs(B, S, H)
    xn = x.cuda().requires_grad_(True)
    set_backend("native")
    try:
        stage = _native_stage(ours)
        stage.train()
        out_n = stage(xn, ext.cuda())[0]
        out_n.backward(cot.cuda().to(out_n.dtype))
    finally:
        set_backend("auto")
    _check_block_against_golden(golden, ours, out_n, xn.grad)


def _check_zero_gradient(layer, key_bias):
    """The key bias has a mathematically ZERO gradient (softmax is invariant to a per-query shift
    of all scores): the reference leaves fp32 round-off there, the bf16 path leaves bf16 round-off;
    require it to be small against the query-bias gradient instead of comparing noise to noise."""
    q = dict(layer.named_parameters())["attention.self.query.bias"].grad
    assert float(key_bias.grad.abs().max()) < 0.1 * float(q.abs().max())


class _FixedMaskDropout(torch.nn.Module):
    """Stands in for nn.Dropout inside the REFERENCE classes: applies a given keep mask."""

    def __init__(self, keep, p):
        super().__init__()
        self.keep, self.p = keep, p

    def forward(self, x):
        return x * self.keep.to(x.dtype).view(x.shape) / (1.0 - self.p)


@pytest.mark.gpu
def test_exact_dropout_mask_parity_with_reference_classes():
    """Dropout ON (p = 0.1): the three masks of a block (attention probabilities, attention
    output, FFN output) are regenerated on the HOST from the dropout RNG state + the sites' stream
    ids and were applied inside the reference's fp32 classes; forward and all gradients must then
    agree like in the dropout-free test (a wrong / shifted mask would give O(1) errors)."""
    from skycomputing_b200.models import default_rng, set_backend
    from skycomputing_b200.ops.dropout_ref import keep_mask

    golden = _golden("dropout")
    torch.manual_seed(0)
    p = 0.1
    cfg = _configs(1024, 16, 4096, p=p, vocab=30522)
    ours = _build_ours(BLOCK, cfg, "cuda")
    assert _state_entries(ours) == list(golden["state"])
    _load_seeded_weights(ours, golden["state"], seed=12, std=0.02)
    B, S, H = 32, 128, 1024
    x, ext, cot = _block_inputs(B, S, H, seed=5)
    xn = x.cuda().requires_grad_(True)
    rng = default_rng(torch.device("cuda", 0))
    saved = rng.state.clone()
    pinned = torch.tensor([DROPOUT_SEED, DROPOUT_STEP], dtype=torch.int64, device=rng.state.device)
    set_backend("native")
    try:
        rng.state.copy_(pinned)
        stage = _native_stage(ours)
        stage.train()
        stage.spans()[0].params.rng_base = DROPOUT_BASE
        out_n = stage(xn, ext.cuda())[0]
        out_n.backward(cot.cuda().to(out_n.dtype))
        assert torch.equal(rng.state, pinned)      # the masks the golden data was computed with
    finally:
        rng.state.copy_(saved)
        set_backend("auto")
    kept = float(keep_mask(DROPOUT_SEED, DROPOUT_STEP, DROPOUT_BASE + 2, (B * S, H), p).mean())
    assert abs(kept - (1 - p)) < 5e-3
    _check_block_against_golden(golden, ours, out_n, xn.grad)


# ------------------------------------------------------------------------------------------------
# golden data: run the reference's classes (fp32, on the CPU) on the inputs above
# ------------------------------------------------------------------------------------------------
def _build_reference(names, cfg, reference):
    for path in (os.path.join(ROOT, "baseline", "stubs"), reference):
        if path not in sys.path:
            sys.path.insert(0, path)
    from scaelum.registry import LAYER as REF_LAYER   # the unmodified reference package

    return [REF_LAYER.get_module(n)(**_layer_kwargs(n, cfg)) for n in names]


def _sample(out, name, t, k, seed):
    flat = t.detach().double().reshape(-1).numpy()
    idx = np.flatnonzero(flat)
    if idx.size > k:
        idx = np.sort(np.random.RandomState(seed).choice(idx, k, replace=False))
    out[name + ".idx"] = idx.astype(np.int32)
    out[name + ".val"] = flat[idx].astype(np.float32)
    out[name + ".norm"] = np.float64(np.linalg.norm(flat))


def _sample_grads(out, layers, k):
    for i, layer in enumerate(layers):
        for n, p in layer.named_parameters():
            if not n.endswith("key.bias"):   # zero in exact arithmetic: see _check_zero_gradient
                _sample(out, f"grad.{i}.{n}", p.grad, k, seed=len(out))


def _make_golden(reference):
    torch.set_num_threads(os.cpu_count() or 1)
    os.makedirs(GOLDEN, exist_ok=True)

    cfg = _configs(64, 4, 128)
    ref = _build_reference(CPU_LAYERS, cfg, reference)
    out = {"state": np.array(_state_entries(ref))}
    _load_seeded_weights(ref, out["state"], seed=10, std=0.1)
    ids, tt, am, cot = _cpu_inputs()
    y = _chain(ref, (ids, tt, am))[0]
    y.backward(cot)
    _sample(out, "out", y, 256, seed=0)
    for i, layer in enumerate(ref):
        for n, p in layer.named_parameters():
            _sample(out, f"grad.{i}.{n}", p.grad, 256, seed=len(out))
    np.savez_compressed(os.path.join(GOLDEN, "reference_oracle_cpu.npz"), **out)

    B, S, H = 32, 128, 1024
    cfg = _configs(1024, 16, 4096, vocab=30522)
    ref = _build_reference(BLOCK * 2, cfg, reference)
    out = {"state": np.array(_state_entries(ref))}
    _load_seeded_weights(ref, out["state"], seed=11, std=0.02)
    x, ext, cot = _block_inputs(B, S, H)
    x.requires_grad_(True)
    for layer in ref:
        layer.eval()                                   # dropout p = 0 anyway
    y = _chain(ref, (x, ext))[0]
    y.backward(cot)
    _sample(out, "out", y, 2048, seed=1)
    _sample(out, "x.grad", x.grad, 2048, seed=2)
    _sample_grads(out, ref, 256)
    np.savez_compressed(os.path.join(GOLDEN, "reference_oracle_block.npz"), **out)

    from skycomputing_b200.ops.dropout_ref import keep_mask

    p, heads = 0.1, 16
    cfg = _configs(1024, 16, 4096, p=p, vocab=30522)
    ref = _build_reference(BLOCK, cfg, reference)
    out = {"state": np.array(_state_entries(ref))}
    _load_seeded_weights(ref, out["state"], seed=12, std=0.02)
    x, ext, cot = _block_inputs(B, S, H, seed=5)
    x.requires_grad_(True)

    def mask(stream, shape):
        return torch.from_numpy(keep_mask(DROPOUT_SEED, DROPOUT_STEP, DROPOUT_BASE + stream, shape, p))

    head, _body, tail = ref
    head.attention.self.dropout = _FixedMaskDropout(mask(1, (B, heads, S, S)), p)
    head.attention.output.dropout = _FixedMaskDropout(mask(2, (B * S, H)), p)
    tail.output.dropout = _FixedMaskDropout(mask(3, (B * S, H)), p)
    y = _chain(ref, (x, ext))[0]
    y.backward(cot)
    _sample(out, "out", y, 2048, seed=1)
    _sample(out, "x.grad", x.grad, 2048, seed=2)
    _sample_grads(out, ref, 256)
    np.savez_compressed(os.path.join(GOLDEN, "reference_oracle_dropout.npz"), **out)


if __name__ == "__main__":
    import argparse

    ap = argparse.ArgumentParser(description="regenerate tests/golden/reference_oracle_*.npz")
    ap.add_argument("--reference", required=True,
                    help="directory that contains the reference's `scaelum` package")
    sys.path.insert(0, ROOT)
    _make_golden(os.path.abspath(ap.parse_args().reference))
