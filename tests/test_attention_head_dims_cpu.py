"""Which head sizes take the native attention path: the Python rule, the fused-boundary negotiation
that follows from it, and the device benchmark's head size (no GPU needed)."""
import pytest

import skycomputing_b200 as sky
from skycomputing_b200.ops import native as nat


@pytest.mark.parametrize("S,d", [(128, 64), (128, 8), (128, 16), (72, 32), (512, 48), (8, 96),
                                 (200, 128), (130 * 8, 120)])
def test_rule_accepts(S, d):
    assert nat.attention_supported(S, d)


@pytest.mark.parametrize("S,d", [(128, 0), (128, 4), (128, 12), (128, 63), (128, 136), (128, 256),
                                 (0, 64), (130, 64), (-8, 64), (127, 32)])
def test_rule_rejects(S, d):
    assert not nat.attention_supported(S, d)


def _block_stage(hidden, heads):
    c = sky.BertConfig(100, hidden_size=hidden, num_hidden_layers=1, num_attention_heads=heads,
                       intermediate_size=2 * hidden, max_position_embeddings=128)
    mc = [dict(layer_type=f"BertLayer_{n}", config=c.__dict__) for n in ("Head", "Body", "Tail")]
    return sky.build_module_from_cfg(0, mc, dict(module_to_cuda=False))


@pytest.mark.parametrize("hidden,heads,fused", [
    (512, 4, True),     # head size 128
    (256, 8, True),     # head size 32
    (1024, 16, True),   # head size 64 (BERT-large)
    (96, 8, False),     # head size 12: not a multiple of 8
    (272, 2, False),    # head size 136: above 128
])
def test_fused_boundary_follows_the_head_size_rule(hidden, heads, fused):
    st = _block_stage(hidden, heads)
    assert st.fused_boundary_support((4, 128, hidden)) == (fused, fused)
    if fused:
        assert st.fused_boundary_support((4, 130, hidden)) == (False, False)   # S % 8 != 0


def test_device_benchmarker_passes_the_head_size(monkeypatch):
    calls = []

    class FakeExt:
        def device_benchmark(self, **kw):
            calls.append(kw)
            return 1.0, 10000.0

    monkeypatch.setattr(nat, "ext", lambda: FakeExt())
    bench = sky.DeviceBenchmarker.local_benchmark_native
    bench({}, 5, 1, dict(tokens=4096, hidden=1024, intermediate=4096))
    bench({}, 5, 1, dict(tokens=4096, hidden=1024, intermediate=4096, head_dim=128))
    bench({}, 5, 1, dict(tokens=4096, hidden=512, intermediate=2048, head_dim=32, heads=8))
    assert [(c["heads"], c["head_dim"]) for c in calls] == [(16, 64), (8, 128), (8, 32)]
