"""tcgen05 attention at head sizes other than 64 (any multiple of 8 up to 128): kernel numerics,
dropout mask parity, the Python support rule, the layer spans and the engines on the native path."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nat():
    from skycomputing_b200.ops import native

    assert native.available(), "native extension must be built and a GPU present"
    return native


def _rand(*shape):
    return torch.randn(*shape, device="cuda", dtype=torch.float32).to(torch.bfloat16)


def _close(got, ref, rtol=2e-2, atol=2e-2):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs().max().item()
    denom = ref.abs().max().item() + 1e-6
    assert torch.isfinite(got).all(), "non-finite output"
    assert err <= atol + rtol * denom, f"max abs err {err} vs ref max {denom}"


def _split(qkv, B, S, heads):
    d = qkv.shape[1] // 3 // heads
    return qkv.float().view(B, S, 3, heads, d).permute(2, 0, 3, 1, 4)


def _attention_ref(qkv, mask, B, S, heads, keep=None, p=0.0):
    H = qkv.shape[1] // 3
    q, k, v = _split(qkv, B, S, heads)
    s = q @ k.transpose(-1, -2) / math.sqrt(H // heads)
    if mask is not None:
        s = s + mask.view(B, 1, 1, S)
    pr = torch.softmax(s, -1)
    if keep is not None:
        pr = pr * keep.to(pr.dtype) / (1.0 - p)
    return (pr @ v).permute(0, 2, 1, 3).reshape(B * S, H)


def _check_grads(dqkv, ref_grad, H):
    _close(dqkv[:, :H], ref_grad[:, :H], rtol=3e-2, atol=3e-2)           # dQ
    _close(dqkv[:, H:2 * H], ref_grad[:, H:2 * H], rtol=3e-2, atol=3e-2)  # dK
    _close(dqkv[:, 2 * H:], ref_grad[:, 2 * H:], rtol=3e-2, atol=3e-2)   # dV


# 48 / 96: a partly padded 64-column block; 8 / 16: mostly padded tiles; 128: two full blocks
@pytest.mark.parametrize("S", [128, 72, 256, 512])
@pytest.mark.parametrize("d", [8, 16, 32, 48, 96, 128])
def test_attention_head_dim_numerics(nat, d, S):
    """Forward, log-sum-exp and all three gradients against the fp32 reference, padding mask."""
    torch.manual_seed(100 + d + S)
    B, heads = 2, 3
    H = heads * d
    assert nat.ext().attention_supported(S, d)
    qkv = _rand(B * S, 3 * H)
    m = torch.ones(B, S, device="cuda")
    m[0, S - S // 4:] = 0
    m[1, S // 2:] = 0
    mask = (1.0 - m) * -10000.0
    ctx, lse = nat.attention_fwd(qkv, mask, B, S, heads)
    qf = qkv.float().requires_grad_(True)
    ref = _attention_ref(qf, mask, B, S, heads)
    _close(ctx, ref)
    q, k, _ = _split(qkv, B, S, heads)
    sc = q @ k.transpose(-1, -2) / math.sqrt(d) + mask.view(B, 1, 1, S)
    lse_ref = torch.logsumexp(sc, -1) / math.log(2.0)
    _close(lse.view(B, heads, S), lse_ref, rtol=1e-3, atol=2e-2)
    dctx = _rand(B * S, H)
    ref.backward(dctx.float())
    dqkv = nat.attention_bwd(qkv, mask, ctx, lse, dctx, B, S, heads)
    _check_grads(dqkv, qf.grad, H)


@pytest.mark.parametrize("S", [128, 256])
@pytest.mark.parametrize("d", [32, 128])
def test_attention_head_dim_dropout_mask_parity(nat, d, S):
    """The host replica of the device RNG gives the exact keep mask; forward and gradients must
    match the fp32 reference that applies it (same element indexing at every head size)."""
    from skycomputing_b200.ops.dropout_ref import keep_mask_from_state

    torch.manual_seed(41 + d)
    B, heads, p = 2, 2, 0.1
    H = heads * d
    rng = nat.RngState(4243)
    qkv = _rand(B * S, 3 * H)
    ctx, lse = nat.attention_fwd(qkv, None, B, S, heads, dropout_p=p, rng=rng, rng_stream=12)
    keep = torch.from_numpy(keep_mask_from_state(rng.state, 12, (B, heads, S, S), p)).cuda()
    qf = qkv.float().requires_grad_(True)
    ref = _attention_ref(qf, None, B, S, heads, keep=keep, p=p)
    _close(ctx, ref)
    dctx = _rand(B * S, H)
    ref.backward(dctx.float())
    dqkv = nat.attention_bwd(qkv, None, ctx, lse, dctx, B, S, heads, dropout_p=p, rng=rng,
                             rng_stream=12)
    _check_grads(dqkv, qf.grad, H)


def test_python_rule_matches_the_kernels(nat):
    for d in range(1, 161):
        for S in (0, 8, 72, 128, 130, 512):
            assert nat.attention_supported(S, d) == nat.ext().attention_supported(S, d), (S, d)
    for d in (12, 136):
        heads = 2
        qkv = _rand(2 * 128, 3 * heads * d)
        with pytest.raises(RuntimeError, match="930"):
            nat.attention_fwd(qkv, None, 2, 128, heads)


@pytest.fixture
def attention_calls(monkeypatch):
    """Counts the calls of the native attention wrappers (ops/functions.py calls them through the
    module, so a shim on the module sees every native span)."""
    from skycomputing_b200.ops import native

    calls = {"fwd": 0, "bwd": 0}
    fwd, bwd = native.attention_fwd, native.attention_bwd

    def counting_fwd(*a, **k):
        calls["fwd"] += 1
        return fwd(*a, **k)

    def counting_bwd(*a, **k):
        calls["bwd"] += 1
        return bwd(*a, **k)

    monkeypatch.setattr(native, "attention_fwd", counting_fwd)
    monkeypatch.setattr(native, "attention_bwd", counting_bwd)
    return calls


@pytest.mark.parametrize("S", [128, 200])
@pytest.mark.parametrize("hidden,heads", [(512, 4), (256, 8)])
def test_layer_span_runs_native_attention(attention_calls, hidden, heads, S):
    """Head + Body + Tail through a ModuleWrapper against the fp32 oracle (forward and every
    parameter gradient); the native span, not the eager fallback, ran the attention."""
    from tests.test_layers_gpu import _cfg, _hidden_inputs, _run_pair

    cfg = _cfg(hidden=hidden, heads=heads, inter=2 * hidden)
    _run_pair(["BertLayer_Head", "BertLayer_Body", "BertLayer_Tail"], _hidden_inputs(cfg, S=S), cfg)
    assert attention_calls == {"fwd": 1, "bwd": 1}


def _d128_model():
    from skycomputing_b200.models import BertConfig

    cfg = BertConfig(1000, hidden_size=512, num_hidden_layers=2, num_attention_heads=4,
                     intermediate_size=1024, max_position_embeddings=128, hidden_dropout_prob=0.0,
                     attention_probs_dropout_prob=0.0)
    block = [dict(layer_type=f"BertLayer_{n}", config=cfg.__dict__) for n in ("Head", "Body", "Tail")]
    return ([dict(layer_type="BertEmbeddings", config=cfg.__dict__)] + block * 2
            + [dict(layer_type="BertPooler", config=cfg.__dict__),
               dict(layer_type="BertTailForClassification", hidden_dropout_prob=0.0,
                    hidden_size=512, num_classes=3)])


def test_single_gpu_engine_captures_head_dim_128(attention_calls):
    """PipelineEngine, one stage, SGD, CUDA graph: 3 eager steps, then capture and replays; the
    first loss matches the eager fp32 model (set_backend("torch")) within the layer-test band."""
    import skycomputing_b200 as sky
    from skycomputing_b200.models import set_backend
    from skycomputing_b200.parallel.pipeline import PipelineEngine

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B, S = 4, 128
    g = torch.Generator(device="cpu").manual_seed(5)
    ids = torch.randint(1000, (B, S), generator=g).cuda()
    tt = torch.zeros(B, S, dtype=torch.long, device=dev)
    mask = torch.ones(B, S, dtype=torch.long, device=dev)
    mask[1, 100:] = 0
    labels = torch.randint(3, (B,), generator=g).cuda()
    loss_fn = sky.build_loss(dict(type="CrossEntropyLoss"), dev)
    try:
        set_backend("torch")
        torch.manual_seed(0)
        ref = sky.build_module_from_cfg(0, _d128_model(), dict(module_to_cuda=True, cuda_device=0))
        with torch.no_grad():
            ref_loss = float(loss_fn(ref(ids, tt, mask)[0], labels))
        assert attention_calls["fwd"] == 0

        set_backend("native")
        torch.manual_seed(0)
        stage = sky.build_module_from_cfg(0, _d128_model(), dict(module_to_cuda=True, cuda_device=0))
        stage.train()
        opt = sky.build_optimizer(stage, dict(optim_type="SGD", lr=1e-3))
        eng = PipelineEngine(stage, 0, 1, [0], dev, opt, loss_fn=loss_fn, micro_batches=1)
        losses = [float(eng.train_step([ids, tt, mask], labels)) for _ in range(5)]
        torch.cuda.synchronize()
    finally:
        set_backend("auto")
    assert eng.graphable and eng._graph is not None
    assert attention_calls["fwd"] >= 2 * 4 and attention_calls["bwd"] >= 2 * 4   # eager + capture
    assert all(math.isfinite(x) for x in losses), losses
    assert losses[0] == pytest.approx(ref_loss, rel=4e-2, abs=4e-2)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_fused_ring_at_head_dim_128():
    """hidden 1024 / 8 heads: both engines negotiate the fused NVLink boundary and capture the
    step; their loss trajectories stay inside the band of the NCCL p2p run."""
    from tests.test_multi_gpu import _run

    common = ("--heads", "8")
    nccl = _run(2, "--boundary", "nccl", *common)
    fused = _run(2, "--boundary", "fused", *common)
    looped = _run(2, "--virtual-stages", "2", *common)
    assert not nccl["fused_any"]
    for r in (fused, looped):
        assert r["fused_any"] and r["graph_all"] and r["err_any"] == 0
        for a, b in zip(r["losses"], nccl["losses"]):
            assert a == pytest.approx(b, rel=3e-3, abs=3e-3)
