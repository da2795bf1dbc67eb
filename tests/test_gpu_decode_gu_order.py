"""The persistent decode kernel's interleaved gate/up unit map (q3_mega.cuh gu_map) on the GPU, in each regime of the map:
F = 0 (fewer than 8 units per CTA: the contiguous split), F = 1 (one interleaved block, then the tail), F >= 2 with a tail
that is not a whole number of quantisation groups, and F >= 2 at group size 128.  F = hidden // num_sms // 8; the regimes
below hold on 148 SMs."""
import os

import numpy as np
import pytest

from qwen3_rs_b200 import synth, transformer as T
from qwen3_rs_b200.sampler import argmax_last

pytestmark = pytest.mark.gpu

# (shape, group size)
CASES = [
    (synth.SHAPES["tiny"], 64),                                                               # hidden 768: F 0
    (synth.SHAPES["small"], 64),                                                              # hidden 1536: F 1
    (synth.Shape("gu-tail32", 256, 3584, 2, 4, 2, vocab_size=1024, max_seq_len=256), 64),     # F 3, tail 32 units = half a group
    (synth.Shape("gu-tail32", 256, 3584, 2, 4, 2, vocab_size=1024, max_seq_len=256), 32),     # F 3, tail 1 group
    (synth.Shape("gu-gs128", 256, 4864, 2, 4, 2, vocab_size=1024, max_seq_len=256), 128),     # F 4, tail 1 group
]
IDS = [f"{s.name}-h{s.hidden_dim}-gs{gs}" for s, gs in CASES]


@pytest.fixture(scope="module", params=range(len(CASES)), ids=IDS)
def model(request, tmp_path_factory):
    shape, gs = CASES[request.param]
    path = os.path.join(str(tmp_path_factory.mktemp("gu")), f"{shape.name}_gs{gs}.bin")
    synth.export_synthetic(shape, path, gs, seed=5)
    m = T.TransformerBuilder.new(path).build()
    try:
        m.set_decode_path(1)
    except T.Q3Error:
        m.close()
        pytest.skip("persistent kernel not available for this shape")
    full = shape.hidden_dim // m.num_sms // 8
    print(f"{IDS[request.param]}: {m.num_sms} SMs, F = {full}, tail {shape.hidden_dim - 8 * m.num_sms * full} units")
    yield m
    m.close()


def test_layerwise_matches_graph_path(model):
    """Same check as the golden shapes' persistent-vs-graph comparison: every layer at round-off except at most one
    attention int8 flip, the head at 1e-4."""
    m = model
    c = m.get_config()
    rng = np.random.default_rng(2)
    errs = []
    try:
        for pos in (0, 3):
            for l in range(c.n_layers):
                x = rng.standard_normal(c.dim).astype(np.float32)
                m.set_decode_path(0)
                a = m.forward_layers(x, pos, l, l + 1)
                m.set_decode_path(1)
                b = m.forward_layers(x, pos, l, l + 1)
                errs.append(float(np.abs(a - b).max()) / max(1.0, float(np.abs(a).max())))
            x = rng.standard_normal(c.dim).astype(np.float32)
            m.set_decode_path(0)
            _, la = m.forward_layers(x, pos, 0, 0, run_head=True)
            m.set_decode_path(1)
            _, lb = m.forward_layers(x, pos, 0, 0, run_head=True)
            assert np.abs(la - lb).max() <= 1e-4 * max(1.0, np.abs(la).max())
        errs = np.sort(np.array(errs))
        assert errs[:-1].max() <= 1e-4 and errs[-1] <= 3e-2
    finally:
        m.set_decode_path(1)


def test_greedy_decode_is_reproducible_and_matches_forward(model):
    """The order in which the SwiGLU words land depends on timing; the values may not.  Two greedy runs through forward()
    give bit-identical logits, and decode_greedy the same tokens."""
    m = model
    runs = []
    for _ in range(2):
        m.reset()
        tok, seq = 3, []
        for p in range(24):
            lg = m.forward(tok, p)
            tok = argmax_last(lg)
            seq.append(tok)
        runs.append((seq, lg.copy()))
    assert runs[0][0] == runs[1][0]
    assert np.array_equal(runs[0][1], runs[1][1])
    for _ in range(2):
        m.reset()
        assert m.decode_greedy(3, 0, 24) == runs[0][0]
