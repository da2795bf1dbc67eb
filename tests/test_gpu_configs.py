"""GPU parity on the shapes BASELINE.json names beyond Qwen3-0.6B: Qwen3-4B (config 3), Qwen3-8B (configs 4-5) incl. a
32 768-row KV cache.  The CPU oracle runs these shapes at 5-9 tokens/s, so the comparisons are a few tokens / one layer.
Checkpoints are synthetic (seeded), generated on the GPU box and quantised by the library's exporter kernel
(byte-identical to the numpy exporter: test_device_quantizer_makes_identical_checkpoints)."""
import os

import numpy as np
import pytest

import bench
from oracle import binding as orc
from qwen3_rs_b200 import transformer as T
from qwen3_rs_b200.sampler import argmax_last
from test_gpu_parity import LOGIT_TOL, check_layerwise, check_prefill_vs_oracle

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


@pytest.fixture(scope="module")
def big():
    cache = {}

    def get(name, ctx):
        key = (name, ctx)
        if key not in cache:
            path = bench.bench_checkpoint(name, 64)
            cache[key] = (T.TransformerBuilder.new(path).with_ctx_length(ctx).build(), path)
        return cache[key]

    yield get
    for m, _ in cache.values():
        m.close()


@pytest.mark.parametrize("name", ["qwen3-4b", "qwen3-8b"])
def test_exact_mode_bit_identical_and_greedy_tokens(big, name):
    """8 greedy tokens: exact mode logits bit-identical to the oracle and the same tokens (BASELINE configs 3-4 shapes)."""
    m, path = big(name, 64)
    orc.set_threads(os.cpu_count() or 1)
    o = orc.Model(path, 64)
    want = o.generate([1], 8)
    o.reset()
    m.set_exact(True)
    try:
        m.reset()
        seq, worst = [1] + want, 0.0
        for pos in range(8):
            lo, lg = o.forward(seq[pos], pos), m.forward(seq[pos], pos)
            worst = max(worst, float(np.abs(lg - lo).max()))
            assert argmax_last(lg) == want[pos]
        print(f"{name} exact mode: 8 greedy tokens identical, max |dlogit| {worst:.2e}")
        assert worst <= 1e-6
    finally:
        m.set_exact(False)
        o.close()


@pytest.mark.parametrize("name", ["qwen3-4b", "qwen3-8b"])
def test_fast_mode_layerwise(big, name):
    """The timed (persistent-kernel) path, layer by layer on the oracle's own residual stream and KV cache."""
    m, path = big(name, 64)
    o, o2 = orc.Model(path, 64), orc.Model(path, 64)
    try:
        check_layerwise(m, o, o2, [1, 43348, 17], name)
    finally:
        o.close()
        o2.close()


def test_8b_attention_over_32k_cache_matches_oracle(big):
    """BASELINE config 5: one Qwen3-8B layer attending over a 32 768-row f32 KV cache (18 splits per kv head in the
    persistent kernel), teacher-forced: injected N(0,1)-scaled K / V rows, the oracle's residual stream in, compared with
    the oracle's residual stream out."""
    npos = 32768
    m, path = big("qwen3-8b", npos + 8)
    o = orc.Model(path, npos + 8)
    try:
        c = o.config
        kv = c["n_kv_heads"] * c["head_dim"]
        rng = np.random.default_rng(8)
        ko, vo = o.kv_cache()
        layer = 1
        # keys small enough that the softmax is not one-hot: thousands of positions carry weight
        ko[layer, :npos] = (rng.standard_normal((npos, c["n_kv_heads"], c["head_dim"])) * 0.3).astype(np.float32)
        vo[layer, :npos] = rng.standard_normal((npos, c["n_kv_heads"], c["head_dim"])).astype(np.float32)
        m.reset()
        for p0 in range(0, npos, 8192):
            m.kv_write(layer, p0, ko[layer, p0:p0 + 8192].reshape(-1, kv), vo[layer, p0:p0 + 8192].reshape(-1, kv))
        x = (rng.standard_normal(c["dim"]) * 0.5).astype(np.float32)
        want = o.forward_layers(x, npos, layer, layer + 1)
        got = m.forward_layers(x, npos, layer, layer + 1)
        err = float(np.abs(got - want).max())
        print(f"8B layer {layer} at pos {npos}: max |dx| {err:.2e} (|x| max {np.abs(want).max():.2f})")
        assert err <= LOGIT_TOL
        k, v = m.kv_read(layer, npos, 1)
        np.testing.assert_allclose(k[0], ko[layer, npos].reshape(-1), rtol=0, atol=1e-4)
        np.testing.assert_allclose(v[0], vo[layer, npos].reshape(-1), rtol=0, atol=1e-4)
    finally:
        o.close()


@pytest.mark.parametrize("name", ["qwen3-4b", "qwen3-8b"])
def test_prefill_2048_prefix_chunk_rerun_invariance_and_oracle(big, name):
    """The bench's prefill workload, T 2048 (up to 21 GEMM tiles per CTA): a rerun, the chunks 1000 + 1048 and a 48-token prefix
    give bit-identical K / V rows of every layer (and logits); the 48-token prefill against the oracle.  Rows 0..47 sit in m-tile 0:
    for n-tile n that is tile 16 n, which a CTA runs on its iteration 16 n / grid, so they cover later tile iterations too."""
    from test_gpu_prefill_scale import assert_same_rows

    m, path = big(name, 4096)
    c = m.get_config()
    toks = np.random.default_rng(7).integers(0, c.vocab_size, 2048).tolist()

    def run(chunks):
        m.reset()
        for a, b in chunks:
            lg = m.prefill(toks[a:b], a)
        return lg

    lg = run([(0, 2048)])
    full = [m.kv_read(l, 0, 2048) for l in range(c.n_layers)]
    for label, chunks in (("rerun", [(0, 2048)]), ("chunks 1000 + 1048", [(0, 1000), (1000, 2048)])):
        lg2 = run(chunks)
        for l in range(c.n_layers):
            assert_same_rows([m.kv_read(l, 0, 2048)], [full[l]], 2048, f"{name} {label} (layer {l})")
        assert np.array_equal(lg2, lg), f"{name} {label}: logits differ"
    run([(0, 48)])
    assert_same_rows([m.kv_read(l, 0, 48) for l in range(c.n_layers)], full, 48, f"{name} 48-token prefix")
    del full
    orc.set_threads(os.cpu_count() or 1)
    check_prefill_vs_oracle(m, path, toks[:48], name, 64)
