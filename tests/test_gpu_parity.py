"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the committed golden vectors.

Tolerances (BASELINE.json north_star): per-group int8 dot products bit-exact; logits max-abs <= 1e-2;
greedy tokens identical.

Two execution modes are tested:
  * exact mode (q3_set_exact): every float reduction in the reference's left-fold order and exp() as
    glibc computes it -> logits are compared at 1e-6 (bit-identical in practice), greedy tokens identical,
    on every golden shape and on the full-size Qwen3-0.6B (BASELINE configs 1-2).
  * fast mode (default, what the bench times): differs from the reference ONLY in the order of float
    sums.  Because the forward pass re-quantises activations to int8 >= 4 times per layer, a last-ulp
    difference can move one int8 by 1, and on random-init weights that single step is amplified by the
    later layers (tests/test_oracle.py::test_reassociation_sensitivity...: the oracle itself moves by
    ~0.7 when only its summation order changes).  Fast mode is therefore held to 1e-2 where no cascade
    exists -- operator level and layer level with teacher-forced inputs (relative to the residual
    stream's scale) -- and end to end against the oracle's own reassociation noise floor.
"""
import numpy as np
import pytest

from conftest import GOLDEN_CASES
from oracle import binding as orc
from qwen3_rs_b200 import generation, transformer as T
from qwen3_rs_b200 import transformer as T_mod
from qwen3_rs_b200.sampler import Sampler, argmax_last

pytestmark = pytest.mark.gpu
LOGIT_TOL = 1e-2  # north_star


# ---- operators ------------------------------------------------------------------------------
@pytest.mark.parametrize("gs", [32, 64, 128])
def test_quantize_bit_exact(gs, golden):
    rng = np.random.default_rng(gs)
    cases = [golden["quant_x"], (rng.standard_normal(12288) * 2).astype(np.float32),
             np.zeros(256, np.float32), (rng.standard_normal(4096) * 1e-20).astype(np.float32)]
    ties = (np.arange(-127, 129, dtype=np.float32) - 0.5)[: 256]
    ties[-1] = 127.0  # scale exactly 1 -> x.5 ties everywhere (round half away from zero)
    cases.append(ties)
    for x in cases:
        q, s = T.op_quantize(x, gs)
        qo, so = orc.quantize(x, gs)
        assert np.array_equal(q, qo) and np.array_equal(s, so)
    q, s = T.op_quantize(golden["quant_x"], gs)
    assert np.array_equal(q, golden[f"quant_q_gs{gs}"]) and np.array_equal(s, golden[f"quant_s_gs{gs}"])


@pytest.mark.parametrize("n,d,gs", [(256, 48, 64), (128, 2, 32), (1024, 2048, 64), (4096, 512, 128), (12288, 64, 64),
                                    (2560, 130, 32), (9728, 34, 64)])
def test_matmul_group_dots_bit_exact(n, d, gs):
    rng = np.random.default_rng(n + d)
    wq = rng.integers(-127, 128, size=d * n, dtype=np.int8)
    wq[:n] = 127  # extreme row: |dot| reaches gs*127*127
    ws = (rng.random(d * n // gs) * 0.02).astype(np.float32)
    x = rng.standard_normal(n).astype(np.float32)
    x[:gs] = np.abs(x[:gs]).max()
    xq, xs = orc.quantize(x, gs)
    out, dots = T.op_matmul(xq, xs, wq, ws, n, d, gs, want_dots=True)
    assert np.array_equal(dots, orc.group_dots(xq, wq, n, d, gs))  # int32, bit-exact
    ref = orc.matmul(xq, xs, wq, ws, n, d, gs)
    # identical per-group terms, only the order of the f32 group sum differs
    scale = np.abs(ref).max() + 1e-30
    assert np.abs(out - ref).max() <= 2e-6 * scale * np.sqrt(n / gs)


def test_matmul_golden(golden):
    out, dots = T.op_matmul(golden["mm_xq"], golden["mm_xs"], golden["mm_wq"], golden["mm_ws"], 256, 48, 64, want_dots=True)
    assert np.array_equal(dots, golden["mm_dots"])
    np.testing.assert_allclose(out, golden["mm_out"], rtol=2e-6, atol=1e-6)


@pytest.mark.parametrize("n,d,gs", [(256, 48, 64), (1024, 512, 64), (4096, 130, 128), (12288, 32, 64), (2560, 66, 32)])
def test_matmul_exact_mode_is_bit_identical(n, d, gs):
    rng = np.random.default_rng(n * 7 + d)
    wq = rng.integers(-127, 128, size=d * n, dtype=np.int8)
    ws = (rng.random(d * n // gs) * 0.02).astype(np.float32)
    xq, xs = orc.quantize(rng.standard_normal(n).astype(np.float32), gs)
    out = T.op_matmul(xq, xs, wq, ws, n, d, gs, exact=True)
    assert np.array_equal(out, orc.matmul(xq, xs, wq, ws, n, d, gs))  # f32, bit for bit


def test_expf_restatement_matches_glibc_bit_for_bit():
    rng = np.random.default_rng(11)
    x = np.concatenate([
        rng.uniform(-104, 89, 1 << 21), rng.uniform(-20, 0, 1 << 21), rng.standard_normal(1 << 20) * 1e-3,
        np.array([0.0, -0.0, 88.72, 88.73, -103.97, -103.98, -87.5, 1e-30, -1e-30, np.inf, -np.inf, 1.0, -1.0]),
    ]).astype(np.float32)
    got, want = T.op_expf(x), orc.expf(x)
    bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))[0]
    assert bad.size == 0, (bad.size, x[bad[:5]], got[bad[:5]], want[bad[:5]])


def test_rmsnorm():
    rng = np.random.default_rng(5)
    for n in (128, 1024, 4096, 2560):
        x = (rng.standard_normal(n) * 3).astype(np.float32)
        w = (1 + 0.1 * rng.standard_normal(n)).astype(np.float32)
        np.testing.assert_allclose(T.op_rmsnorm(x, w), orc.rmsnorm(x, w), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("gs", [32, 64, 128])
def test_exporter_quantizer_on_device_bit_exact(gs):
    rng = np.random.default_rng(9)
    w = (rng.standard_normal(1 << 18) * 0.05).astype(np.float32)
    w[:gs] = 0
    w[gs:2 * gs] = np.arange(gs, dtype=np.float32) * 0.5  # exact .5 ties -> half to even
    w[2 * gs - 1] = 127.0
    w[5 * gs + 3] = np.nan
    q, s, _ = T.op_quantize_q80(w, gs)
    qo, so, _ = orc.quantize_q80(w, gs)
    assert np.array_equal(q, qo) and np.array_equal(s, so)
    q, s, _ = T.op_quantize_q80(np.float32([0.0, 127.0, -127.0, 63.5] + [0.0] * (gs - 4)), gs)
    assert q[:4].tolist() == [0, 127, -127, 64] and s[0] == 1.0  # model_exporter_test.rs:48-67


# ---- whole model, small golden shapes ---------------------------------------------------------
@pytest.fixture(scope="module")
def models(ckpt):
    cache = {}

    def get(name, gs, seed, ctx=None):
        key = (name, gs, seed, ctx)
        if key not in cache:
            cache[key] = T.TransformerBuilder.new(ckpt(name, gs, seed)).with_ctx_length(ctx).build()
        return cache[key]

    yield get
    for m in cache.values():
        m.close()


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_config_matches(models, ckpt, name, gs, seed):
    g = models(name, gs, seed).get_config()
    o = orc.Model(ckpt(name, gs, seed)).config
    for k, v in o.items():
        assert int(getattr(g, k)) == v


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_exact_mode_logits_match_golden(models, golden, name, gs, seed):
    """Reference-order CUDA path vs the committed oracle logits: 1e-6 (expected: bit-identical)."""
    key = f"{name}_gs{gs}"
    m = models(name, gs, seed)
    m.set_exact(True)
    try:
        m.reset()
        seq = golden[key + "_prompt"].tolist() + golden[key + "_greedy"].tolist()
        lg = golden[key + "_logits"]
        for p in range(lg.shape[0]):
            out = m.forward(seq[p], p)
            np.testing.assert_allclose(out, lg[p], rtol=0, atol=1e-6)
            assert argmax_last(out) == argmax_last(lg[p])
    finally:
        m.set_exact(False)


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_exact_mode_greedy_tokens_identical_to_golden(models, golden, name, gs, seed):
    key = f"{name}_gs{gs}"
    m = models(name, gs, seed)
    m.set_exact(True)
    try:
        m.reset()
        prompt, want = golden[key + "_prompt"].tolist(), golden[key + "_greedy"].tolist()
        got = generation.generate(m, Sampler(m.get_config().vocab_size, 0.0, 0.9, 0), prompt, len(want))
        assert got == want
        m.reset()
        assert generation.generate_fast(m, prompt, len(want)) == want  # device-resident loop
    finally:
        m.set_exact(False)


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_fast_mode_logits_vs_golden(models, golden, name, gs, seed):
    """Fast mode, teacher-forced along the golden sequence.  Until an int8 activation flips the error is
    float round-off (<< 1e-2); after a flip it is bounded by the cascade noise (the layer-level test
    below is the sharp one).  Required: every position within the noise bound, same argmax wherever the
    golden top-2 margin exceeds twice the observed error."""
    key = f"{name}_gs{gs}"
    m = models(name, gs, seed)
    m.reset()
    seq = golden[key + "_prompt"].tolist() + golden[key + "_greedy"].tolist()
    lg = golden[key + "_logits"]
    errs = []
    for p in range(lg.shape[0]):
        out = m.forward(seq[p], p)
        err = float(np.abs(out - lg[p]).max())
        errs.append(err)
        top2 = np.sort(lg[p])[-2:]
        if top2[1] - top2[0] > 2 * err:
            assert argmax_last(out) == argmax_last(lg[p])
    print(f"{key}: fast-mode max|dlogit| per position {np.array2string(np.array(errs), precision=2)}")
    assert max(errs) <= 0.05 * float(np.abs(lg).max()) + LOGIT_TOL


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_fast_mode_layerwise_matches_oracle(models, ckpt, name, gs, seed):
    m, o = models(name, gs, seed), orc.Model(ckpt(name, gs, seed))
    check_layerwise(m, o, orc.Model(ckpt(name, gs, seed)), [5, 9, 2, 7, 1, 3])


def check_layerwise(m, o, o2, tokens, label=""):
    """Fast mode, one layer at a time, each fed the oracle's own residual stream and KV cache (teacher
    forcing, so nothing cascades).  Without an int8 flip a layer agrees to float round-off; with one
    (a value within an ulp of a rounding boundary landing on the other side) the layer output moves by
    about one quantisation step times a weight.  The yardstick is the oracle itself re-run with
    re-associated sums (perturb mode): the GPU must agree with the oracle as well as the oracle agrees
    with its own re-association -- median at round-off level, worst case within 3x, and the logits
    computed from the oracle's final residual within the north-star 1e-2."""
    gpu_x, gpu_lg = layerwise_errors(m, o, tokens, exact=False)
    ref_x, ref_lg = layerwise_errors(OracleAsModel(o2), o, tokens, exact=False)
    print(f"{label} layerwise |dx|/scale: gpu median {np.median(gpu_x):.2e} worst {gpu_x.max():.2e} "
          f"(>1e-3: {np.mean(gpu_x > 1e-3):.0%}); oracle re-association median {np.median(ref_x):.2e} "
          f"worst {ref_x.max():.2e} (>1e-3: {np.mean(ref_x > 1e-3):.0%}); |dlogit| gpu {gpu_lg:.2e} ref {ref_lg:.2e}")
    # median: at round-off, unless the oracle's own re-association is not (2 layers of a 5120-wide synthetic model: layer 0
    # flips an int8 activation at almost every position, see check_prefill_vs_oracle)
    assert np.median(gpu_x) <= max(1e-5, 3 * np.median(ref_x))
    assert gpu_x.max() <= 3 * ref_x.max() + 1e-3
    assert gpu_lg <= LOGIT_TOL


class OracleAsModel:
    """The oracle in perturb mode (re-associated float sums) behind the Transformer test surface."""

    def __init__(self, o):
        self.o = o

    def reset(self):
        self.o.reset()

    def set_exact(self, on):
        pass

    def kv_write(self, layer, pos0, k, v):
        kc, vc = self.o.kv_cache()
        n = k.shape[0]
        kc[layer, pos0:pos0 + n] = k.reshape(n, kc.shape[2], kc.shape[3])
        vc[layer, pos0:pos0 + n] = v.reshape(n, kc.shape[2], kc.shape[3])

    def forward_layers(self, x, pos, l0, l1, run_head=False):
        orc.set_perturb(1)
        try:
            return self.o.forward_layers(x, pos, l0, l1, run_head)
        finally:
            orc.set_perturb(0)


def layerwise_errors(m, o, tokens, exact):
    """Teacher-forced layer-by-layer comparison against oracle `o`.
    Returns (array of |dx|inf / max(1, |x|inf) per (pos, layer), worst |dlogit|)."""
    c = o.config
    kv = c["n_kv_heads"] * c["head_dim"]
    o.reset()
    m.reset()
    m.set_exact(exact)
    xd = o.dump_residuals()
    errs, worst_lg = [], 0.0
    try:
        for pos, tok in enumerate(tokens):
            lo = o.forward(tok, pos)
            ko, vo = o.kv_cache()
            for l in range(c["n_layers"]):
                m.kv_write(l, 0, ko[l, :pos + 1].reshape(pos + 1, kv), vo[l, :pos + 1].reshape(pos + 1, kv))
                x = m.forward_layers(xd[l], pos, l, l + 1)
                scale = max(1.0, float(np.abs(xd[l + 1]).max()))
                errs.append(float(np.abs(x - xd[l + 1]).max()) / scale)
            _, lg = m.forward_layers(xd[c["n_layers"]], pos, 0, 0, run_head=True)
            worst_lg = max(worst_lg, float(np.abs(lg - lo).max()))
    finally:
        m.set_exact(False)
    return np.array(errs), worst_lg


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_persistent_kernel_matches_graph_path_layerwise(models, name, gs, seed):
    """The single-launch persistent decode kernel vs the multi-kernel CUDA graph on identical inputs: the same per-group terms and
    element-wise operations, so every layer (and the head) agrees to float round-off -- except that the two attention loops add
    in different orders (persistent kernel: lane = cached position, one softmax update per 32 positions), so once in a while an
    attention output lands on the other side of an int8 rounding boundary and that one layer differs by a quantisation step
    (~1e-3 of its scale).  At most one such case per model is accepted here; everything else must be at round-off."""
    m = models(name, gs, seed)
    c = m.get_config()
    rng = np.random.default_rng(1)
    try:
        m.set_decode_path(1)
    except T.Q3Error:
        pytest.skip("persistent kernel not available for this shape")
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
        print(f"{name} gs{gs}: persistent vs graph path, layer-wise |dx|/scale sorted: {np.array2string(errs, precision=1)}")
        assert errs[:-1].max() <= 1e-4 and errs[-1] <= 3e-2
    finally:
        m.set_decode_path(1)


def test_persistent_attention_splits_match_graph_path(models):
    """Attention over a filled cache on both sides of every split boundary of the persistent kernel (one (kv head, split)
    work item per CTA, 32 positions per split, merged by the o_proj prologue): same layer output as the graph path's
    split-K kernels up to float round-off."""
    m = models("small", 64, 3)
    c = m.get_config()
    kvd = c.n_kv_heads * c.head_dim
    rng = np.random.default_rng(5)
    m.reset()
    for l in range(c.n_layers):
        m.kv_write(l, 0, rng.standard_normal((c.seq_len, kvd)).astype(np.float32), rng.standard_normal((c.seq_len, kvd)).astype(np.float32))
    try:
        for pos in (31, 32, 33, 63, 64, 65, 130, 299, c.seq_len - 1):
            x = rng.standard_normal(c.dim).astype(np.float32)
            m.set_decode_path(0)
            a = m.forward_layers(x, pos, 1, 2)
            m.set_decode_path(1)
            b = m.forward_layers(x, pos, 1, 2)
            assert np.abs(a - b).max() <= 1e-4 * max(1.0, np.abs(a).max()), pos
    finally:
        m.set_decode_path(1)
        m.reset()


def test_kv_cache_rows_match_oracle(models, ckpt):
    name, gs, seed = "tiny-untied", 64, 1
    m, o = models(name, gs, seed), orc.Model(ckpt(name, gs, seed))
    m.reset()
    toks = [9, 2, 200, 113]
    for p, t in enumerate(toks):
        m.forward(t, p)
        o.forward(t, p)
    ko, vo = o.kv_cache()
    for l in range(o.config["n_layers"]):
        k, v = m.kv_read(l, 0, len(toks))
        np.testing.assert_allclose(k, ko[l, :len(toks)].reshape(len(toks), -1), rtol=0, atol=1e-4)
        np.testing.assert_allclose(v, vo[l, :len(toks)].reshape(len(toks), -1), rtol=0, atol=1e-4)
        k, v = m.kv_read(l, len(toks), 2)
        assert not k.any() and not v.any()  # untouched rows stay zero (qwen3.rs:439-440)


def test_forward_argmax_and_decode_greedy_agree_with_forward(models):
    m = models("tiny-untied", 64, 1)
    m.reset()
    tok, seq = 9, []
    for p in range(10):
        tok = argmax_last(m.forward(tok, p))
        seq.append(tok)
    m.reset()
    tok, seq2 = 9, []
    for p in range(10):
        tok = m.forward_argmax(tok, p)
        seq2.append(tok)
    m.reset()
    assert seq == seq2 == m.decode_greedy(9, 0, 10)


def test_bounds_are_errors_not_ub(models):
    m = models("micro", 32, 7)
    c = m.get_config()
    for tok, pos in [(c.vocab_size, 0), (-1, 0), (0, c.seq_len), (0, -1)]:
        with pytest.raises(T.Q3Error) as e:
            m.forward(tok, pos)
        assert e.value.code == -1 and "index out of bounds" in e.value.message
    # prompts: a token id outside the vocabulary, and positions pos0 .. pos0+n-1 running past the context
    for toks, pos0 in [([1, c.vocab_size], 0), ([-1, 1], 0), ([1, 2], c.seq_len - 1)]:
        for run in (m.prefill, m.bench_prefill, m.score):
            with pytest.raises(T.Q3Error) as e:
                run(toks, pos0=pos0)
            assert e.value.code == -1 and "index out of bounds" in e.value.message, run.__name__
    m.forward(1, 0)


def test_ctx_length_override(models):
    m = models("tiny", 64, 0, 32)
    assert m.get_config().seq_len == 32  # models/mod.rs:65-67
    with pytest.raises(T.Q3Error):
        m.forward(0, 32)


def test_long_context_split_k_attention_matches_oracle(models, ckpt):
    """Past 128 positions the attention kernel splits the sequence across CTAs; compare layer by layer
    with the oracle's cache injected (teacher forcing) at pos 300 of a 512-token context."""
    name, gs, seed = "small", 128, 2
    m, o = models(name, gs, seed), orc.Model(ckpt(name, gs, seed))
    c = o.config
    rng = np.random.default_rng(3)
    pos = 300
    kv = c["n_kv_heads"] * c["head_dim"]
    ko, vo = o.kv_cache()
    ko[:, :pos] = rng.standard_normal((c["n_layers"], pos, c["n_kv_heads"], c["head_dim"])).astype(np.float32)
    vo[:, :pos] = rng.standard_normal((c["n_layers"], pos, c["n_kv_heads"], c["head_dim"])).astype(np.float32)
    m.reset()
    for l in range(c["n_layers"]):
        m.kv_write(l, 0, ko[l, :pos].reshape(pos, kv), vo[l, :pos].reshape(pos, kv))
    xd = o.dump_residuals()
    lo = o.forward(17, pos)
    for l in range(c["n_layers"]):
        x = m.forward_layers(xd[l], pos, l, l + 1)
        assert np.abs(x - xd[l + 1]).max() <= LOGIT_TOL
    _, lg = m.forward_layers(xd[c["n_layers"]], pos, 0, 0, run_head=True)
    assert np.abs(lg - lo).max() <= LOGIT_TOL


# ---- BASELINE.json config 2: Qwen3-0.6B Q8 gs64 ---------------------------------------------------
@pytest.fixture(scope="module")
def q06(ckpt):
    path = ckpt("qwen3-0.6b", 64, 0)
    m = T.TransformerBuilder.new(path).with_ctx_length(256).build()
    o = orc.Model(path, 256)
    yield m, o
    m.close()


@pytest.mark.slow
def test_qwen3_06b_exact_mode_greedy_128_identical_and_logits_bit_level(q06):
    """BASELINE configs 1-2: Qwen3-0.6B gs64, 128 greedy tokens.  Exact mode reproduces the CPU reference
    run token for token, with logits within 1e-6 at sampled steps."""
    m, o = q06
    o.reset()
    want, margins = o.generate([1], 128, with_margins=True)
    m.set_exact(True)
    try:
        m.reset()
        got = generation.generate_fast(m, [1], 128)
        assert got == want
        o.reset()
        m.reset()
        seq = [1] + want
        worst = 0.0
        for pos in range(24):
            lo, lg = o.forward(seq[pos], pos), m.forward(seq[pos], pos)
            worst = max(worst, float(np.abs(lg - lo).max()))
        print(f"0.6B exact mode: 128 greedy tokens identical (oracle min margin {margins.min():.4f}); "
              f"max |dlogit| over 24 teacher-forced steps {worst:.2e}")
        assert worst <= 1e-6
    finally:
        m.set_exact(False)


@pytest.mark.slow
def test_qwen3_06b_fast_mode_layerwise_parity(q06, ckpt):
    """Every layer of the full-size model, fed the oracle's residual stream and KV cache."""
    m, o = q06
    check_layerwise(m, o, orc.Model(ckpt("qwen3-0.6b", 64, 0), 256), [1, 43348, 17, 99, 5], "0.6B")


@pytest.mark.slow
def test_qwen3_06b_fast_mode_free_running_vs_noise_floor(q06, ckpt):
    """Free-running fast mode along the oracle's greedy sequence: GPU-vs-oracle logit error next to the
    oracle's own error when only ITS summation order changes.  The GPU must stay within 3x that noise
    floor and pick the same token wherever the oracle's top-2 margin exceeds twice the GPU error."""
    m, o = q06
    o.reset()
    toks, margins = o.generate([1], 64, with_margins=True)
    seq = [1] + toks
    o.reset()
    m.reset()
    noise = orc.Model(ckpt("qwen3-0.6b", 64, 0), 256)
    gpu_err, noise_err, mism, agree = [], [], 0, 0
    for pos in range(64):
        lo = o.forward(seq[pos], pos)
        lg = m.forward(seq[pos], pos)
        orc.set_perturb(1)
        try:
            ln = noise.forward(seq[pos], pos)
        finally:
            orc.set_perturb(0)
        gpu_err.append(float(np.abs(lg - lo).max()))
        noise_err.append(float(np.abs(ln - lo).max()))
        agree += argmax_last(lg) == toks[pos]
        if margins[pos] > 2 * gpu_err[-1] and argmax_last(lg) != toks[pos]:
            mism += 1
    print(f"0.6B fast mode free-running: max|dlogit| median {np.median(gpu_err):.3f} max {max(gpu_err):.3f}; "
          f"oracle reassociation noise median {np.median(noise_err):.3f} max {max(noise_err):.3f}; "
          f"argmax agreement {agree}/64")
    assert mism == 0
    assert np.median(gpu_err) <= 3 * np.median(noise_err) + LOGIT_TOL


def test_chat_turns_through_one_prefill_each(models):
    """generation.chat (the reference's chat loop on token ids) with one q3_prefill per user turn: positions, KV rows
    and sampler RNG advance exactly as the reference's token-by-token loop; the first reply token agrees whenever
    the sequential path's top-2 margin is wider than the fast-mode noise."""
    m = models("small", 64, 3)
    V = m.get_config().vocab_size
    turns = [[5, 9, 200, 31, 77, 3], [7, 7, 300]]
    m.reset()
    sa = Sampler(V, 0.8, 0.9, 7)
    ra = generation.chat(m, sa, turns, use_prefill=False, max_new_per_turn=4)
    kv_a = m.kv_read(0, 0, 17)
    m.reset()
    sb = Sampler(V, 0.8, 0.9, 7)
    rb = generation.chat(m, sb, turns, use_prefill=True, max_new_per_turn=4)
    kv_b = m.kv_read(0, 0, 17)
    assert [len(r) for r in ra] == [len(r) for r in rb] == [4, 4]
    assert sa.rng_state == sb.rng_state  # same number of draws
    # layer-0 K/V rows of the first turn depend only on the tokens: identical up to reassociation
    np.testing.assert_allclose(kv_b[0][:6], kv_a[0][:6], rtol=0, atol=2e-3)
    np.testing.assert_allclose(kv_b[1][:6], kv_a[1][:6], rtol=0, atol=2e-3)
    m.reset()
    for p, t in enumerate(turns[0]):
        lg = m.forward(t, p)
    top = np.sort(lg)[-2:]
    m.reset()
    g1 = generation.chat(m, Sampler(V, 0.0, 0.9, 0), turns[:1], use_prefill=True, max_new_per_turn=1)[0]
    if top[1] - top[0] > 0.5:
        assert g1 == [argmax_last(lg)]


# ---- batched prefill: tcgen05 int8 GEMM -----------------------------------------------------------
@pytest.mark.parametrize("T,N,K,gs", [(128, 128, 128, 64), (37, 256, 512, 64), (300, 384, 1024, 32), (130, 128, 2560, 128),
                                      (257, 512, 4096, 64)])
def test_tensor_core_gemm_bit_identical_to_reference_matmul(T, N, K, gs):
    """tcgen05.mma.kind::i8 with per-group TMEM drains: every output equals the oracle's per-token matmul
    bit for bit (exact int32 group dots, identical f32 terms, groups added in order)."""
    rng = np.random.default_rng(T + N + K)
    wq = rng.integers(-127, 128, size=N * K, dtype=np.int8)
    ws = (rng.random(N * K // gs) * 0.02).astype(np.float32)
    xq = np.empty((T, K), np.int8)
    xs = np.empty((T, K // gs), np.float32)
    for t in range(T):
        xq[t], xs[t] = orc.quantize(rng.standard_normal(K).astype(np.float32) * (1 + t % 3), gs)
    xq[0, :] = 127  # extreme row
    wq[:K] = -127
    out = T_mod.op_gemm_q8(xq, xs, wq, ws, T, N, K, gs, exact=True)
    ref = np.stack([orc.matmul(xq[t], xs[t], wq, ws, K, N, gs) for t in range(T)])
    assert np.array_equal(out, ref), float(np.abs(out - ref).max())
    # the drain q3_prefill runs: same int32 group dots and group order, fused multiply-adds -> float round-off of the fold only
    fast = T_mod.op_gemm_q8(xq, xs, wq, ws, T, N, K, gs)
    scale = np.abs(ref).max() + 1e-30
    assert np.abs(fast - ref).max() <= 2e-6 * scale * np.sqrt(K / gs)


def test_tensor_core_gemm_rejects_unknown_modes():
    """The GEMM has two drains, fast (0) and exact (1); any other mode is an argument error, not a different computation."""
    T, N, K, gs = 128, 128, 128, 64
    xq, wq = np.zeros((T, K), np.int8), np.zeros(N * K, np.int8)
    xs, ws = np.ones((T, K // gs), np.float32), np.ones(N * K // gs, np.float32)
    for mode in (2, 5, -1):
        with pytest.raises(T_mod.Q3Error) as e:
            T_mod.op_gemm_q8(xq, xs, wq, ws, T, N, K, gs, exact=mode)
        assert e.value.code == -1  # Q3_EINVAL
        with pytest.raises(T_mod.Q3Error) as e:
            T_mod.bench_gemm_q8(T, N, K, gs, mode, 1)
        assert e.value.code == -1


@pytest.mark.parametrize("name,gs,seed,T", [("tiny-untied", 64, 1, 37), ("small", 128, 2, 130), ("tiny", 64, 0, 5)])
def test_prefill_matches_sequential_forwards(models, name, gs, seed, T):
    """q3_prefill (batched tensor-core path) leaves the KV cache and the last-token logits as T sequential
    forwards would, up to fast-mode float reassociation."""
    m = models(name, gs, seed)
    c = m.get_config()
    rng = np.random.default_rng(T)
    toks = rng.integers(0, c.vocab_size, T).tolist()
    m.reset()
    for p, t in enumerate(toks):
        lg_seq = m.forward(t, p)
    kv_seq = [m.kv_read(l, 0, T) for l in range(c.n_layers)]
    m.reset()
    lg_pf = m.prefill(toks, 0)
    kv_pf = [m.kv_read(l, 0, T) for l in range(c.n_layers)]
    # layer 0 depends only on embedding -> norm -> QKV GEMM -> QK-norm/RoPE: no cascade possible
    np.testing.assert_allclose(kv_pf[0][0], kv_seq[0][0], rtol=0, atol=2e-3)
    np.testing.assert_allclose(kv_pf[0][1], kv_seq[0][1], rtol=0, atol=2e-3)
    assert np.median(np.abs(kv_pf[0][1] - kv_seq[0][1])) <= 1e-6
    for l in range(c.n_layers):
        assert np.abs(kv_pf[l][1] - kv_seq[l][1]).max() <= 0.05 * np.abs(kv_seq[l][1]).max() + 1e-2
        k, v = m.kv_read(l, T, 1)
        assert not k.any() and not v.any()
    err = float(np.abs(lg_pf - lg_seq).max())
    print(f"{name} prefill T={T}: max|dlogit| {err:.2e}")
    assert err <= 0.05 * float(np.abs(lg_seq).max()) + LOGIT_TOL
    # decode continues seamlessly from the prefilled cache
    nxt = argmax_last(lg_pf)
    a = m.forward(nxt, T)
    assert np.isfinite(a).all()


# ---- round 2: bench checkpoints, epoch wrap, reduction-order attribution switches ------------------
def test_device_quantizer_makes_identical_checkpoints(tmp_path):
    """bench.py / the big-config tests quantise their synthetic checkpoints with the library's own exporter kernel
    (k_quantize_q80 on device buffers): the .bin must be byte-identical to the numpy exporter's."""
    import torch

    from qwen3_rs_b200 import synth

    a, b = str(tmp_path / "cpu.bin"), str(tmp_path / "dev.bin")
    for name, gs in (("tiny-untied", 64), ("small", 32)):
        synth.export_synthetic(synth.SHAPES[name], a, gs, seed=5)
        synth.export_synthetic(synth.SHAPES[name], b, gs, seed=5, device="cuda", quantizer=synth.quantize_q80_device)
        da, db = open(a, "rb").read(), open(b, "rb").read()
        if da != db:
            # torch's CUDA and CPU generators differ: compare the quantiser on identical floats instead
            t = synth.make_tensor("model.layers.0.mlp.up_proj.weight", (512, 256), "linear", 5, device="cuda")
            q1, s1, _ = synth.quantize_q80_device(t, gs)
            q0, s0, _ = orc.quantize_q80(t.cpu().numpy(), gs)
            assert np.array_equal(q0, q1) and np.array_equal(s0, s1)
    rng = np.random.default_rng(3)
    w = (rng.standard_normal(1 << 20) * 0.03).astype(np.float32)
    w[:64] = 0.0
    w[64:128] = np.arange(64, dtype=np.float32) * 0.5
    w[127] = 127.0
    for gs in (32, 64, 128):
        q1, s1, _ = synth.quantize_q80_device(torch.from_numpy(w).cuda(), gs)
        q0, s0, _ = orc.quantize_q80(w, gs)
        assert np.array_equal(q0, q1) and np.array_equal(s0, s1)


def test_flagged_exchange_epoch_wraparound(models):
    """The persistent kernel's (payload, epoch) words use epochs = (exchanges issued mod 2^32 - 1) + 1.  Put the counter
    just below the wrap so that it wraps in the middle of a token: same tokens and logits as a fresh run."""
    m = models("small", 64, 3)
    m.reset()
    want = m.decode_greedy(9, 0, 12)
    lg_want = m.forward(want[-1], 12)
    L = m.get_config().n_layers
    for off in (3, 6 * L // 2 + 1, 6 * L * 3 + 2):
        m.reset()
        m.debug_set_epoch(0xFFFFFFFF - off)
        assert m.decode_greedy(9, 0, 12) == want
        assert np.array_equal(m.forward(want[-1], 12), lg_want)


def test_exact_mask_switches_one_reduction_at_a_time(models, golden):
    """q3_set_exact_mask: all five reference-order switches together are exact mode (bit-identical logits); each alone
    still runs and stays inside the fast-mode envelope."""
    name, gs, seed = "tiny-untied", 64, 1
    key = f"{name}_gs{gs}"
    m = models(name, gs, seed)
    seq = golden[key + "_prompt"].tolist() + golden[key + "_greedy"].tolist()
    lg = golden[key + "_logits"]
    try:
        for mask in (31, 1, 2, 4, 8, 16):
            m.set_exact_mask(mask)
            m.reset()
            err = max(float(np.abs(m.forward(seq[p], p) - lg[p]).max()) for p in range(4))
            if mask == 31:
                assert err <= 1e-6
            else:
                assert err <= 0.05 * float(np.abs(lg).max()) + LOGIT_TOL
    finally:
        m.set_exact(False)


@pytest.mark.parametrize("name,gs,seed,T", [("tiny-untied", 64, 1, 37), ("small", 128, 2, 130), ("small", 64, 3, 200)])
def test_prefill_matches_oracle(models, ckpt, name, gs, seed, T):
    """q3_prefill (tcgen05 GEMMs + tensor-core attention) against the ORACLE's T sequential forwards: K / V cache rows of
    every layer and the logits of the last token.  Layer 0 depends only on embedding -> norm -> QKV GEMM -> QK-norm / RoPE
    (nothing can cascade): 1e-4.  Deeper layers see the attention output re-quantised to int8: most rows agree to float
    round-off (median), a flipped int8 moves a row by a quantisation step, bounded by the fast-mode envelope."""
    m = models(name, gs, seed)
    rng = np.random.default_rng(T + 1)
    check_prefill_vs_oracle(m, ckpt(name, gs, seed), rng.integers(0, m.get_config().vocab_size, T).tolist(), f"{name} gs{gs}")


def check_prefill_vs_oracle(m, path, toks, label, ctx=None):
    """The checks of test_prefill_matches_oracle for model `m` against the oracle of checkpoint `path` on prompt `toks`."""
    o, o2 = orc.Model(path, ctx), orc.Model(path, ctx)
    try:
        _check_prefill_vs_oracle(m, o, o2, toks, label)
    finally:
        o.close()
        o2.close()


def _check_prefill_vs_oracle(m, o, o2, toks, label):
    c = o.config
    T = len(toks)
    o.reset()
    o2.reset()
    xd = o.dump_residuals()
    for p, t in enumerate(toks):
        lo = o.forward(t, p)
        orc.set_perturb(1)  # the oracle's own re-association noise on layer 0: o2 runs it on the same embedding row, sums re-associated
        try:
            o2.forward_layers(xd[0], p, 0, 1)
        finally:
            orc.set_perturb(0)
    ko, vo = o.kv_cache()
    ko2, vo2 = o2.kv_cache()
    m.reset()
    lg = m.prefill(toks, 0)
    kvd = c["n_kv_heads"] * c["head_dim"]
    for l in range(c["n_layers"]):
        k, v = m.kv_read(l, 0, T)
        kr, vr = ko[l, :T].reshape(T, kvd), vo[l, :T].reshape(T, kvd)
        ek, ev = np.abs(k - kr), np.abs(v - vr)
        if l == 0:  # embedding -> norm -> quantise -> QKV GEMM -> QK-norm / RoPE: exact up to float round-off, except in the token
            # whose RMSNorm sum lands an ulp off the oracle's and flips an int8 activation (a row then moves by ~1e-3 .. 1e-2).
            # Layer 0 of the SYNTHETIC checkpoints is the worst case for that: the input is int8 x scale (the embedding row) times a
            # bf16-rounded norm weight, so x / scale lands on exact .5 ties far more often than real activations do -- up to 18 % of
            # the rows here (24 / 130 on small gs128, 60 / 200 on small gs64; the sequential decode path flips the very same rows:
            # scripts/diag/prefill_rows.py).  On the CPU alone (scripts/diag/layer0_ties.py, tests/test_oracle.py): 57 % of these
            # rows hold an element within 1e-6 of a tie, and moving the normalisation factor by ONE ulp changes 23 % of them.
            # A row flips when ANY of its dim elements does, so the share of such rows grows with the width (dim 512: <= 30 %,
            # 2560 .. 5120: 75 .. 95 %) -- and with it the median error.  The yardstick is therefore the oracle itself with
            # re-associated sums (o2): the GPU must not flip more rows, nor by more, than that does (and never more than a step).
            ek2 = np.abs(ko2[0, :T].reshape(T, kvd) - kr)
            ev2 = np.abs(vo2[0, :T].reshape(T, kvd) - vr)
            rows_off, rows_ref = float(np.mean(ek.max(axis=1) > 1e-4)), float(np.mean(ek2.max(axis=1) > 1e-4))
            print(f"{label} prefill layer 0: rows off the oracle {rows_off:.0%} (oracle re-association {rows_ref:.0%}), median |dK| "
                  f"{np.median(ek):.1e} ({np.median(ek2):.1e}), max {ek.max():.1e} ({ek2.max():.1e})")
            assert np.median(ek) <= max(1e-6, 3 * np.median(ek2)) and np.median(ev) <= max(1e-6, 3 * np.median(ev2)), label
            assert rows_off <= max(0.4, 1.25 * rows_ref) and ek.max() <= 2e-2, (rows_off, rows_ref, float(ek.max()))
        # deeper layers: an upstream flip perturbs every later element a little (and, through attention, later tokens), so only the
        # noise level is checked here -- the attention kernel itself is compared with float64 in test_prefill_attention_against_float64
        assert np.median(ev) <= 1e-2 * max(1.0, float(np.abs(vr).max())), (l, float(np.median(ev)))
        assert ev.max() <= 0.05 * np.abs(vr).max() + 1e-2 and ek.max() <= 0.05 * np.abs(kr).max() + 1e-2
        k1, v1 = m.kv_read(l, T, 1)
        assert not k1.any() and not v1.any()
    err = float(np.abs(lg - lo).max())
    print(f"{label} prefill T={T} vs oracle: max|dlogit| {err:.2e} (|logit| max {np.abs(lo).max():.1f})")
    assert err <= 0.05 * float(np.abs(lo).max()) + LOGIT_TOL


@pytest.mark.parametrize("T,pos0,n_heads,n_kv", [(70, 0, 8, 2), (33, 45, 4, 4), (129, 3, 16, 2), (200, 0, 2, 1),
                                                 (1000, 1100, 40, 5), (517, 1531, 16, 8),
                                                 pytest.param(2048, 0, 32, 8, marks=pytest.mark.slow)])
def test_prefill_attention_against_float64(T, pos0, n_heads, n_kv):
    """The batched causal attention alone (the tensor-core kernel q3_prefill runs, FP16 hi / lo split) against a float64
    softmax attention: f32-class accuracy (1e-5 of the value scale), i.e. the operand split loses nothing that matters to the
    int8 re-quantisation behind it."""
    rng = np.random.default_rng(T + pos0)
    hd, nk = 128, pos0 + T
    q = rng.standard_normal((T, n_heads * hd)).astype(np.float32)
    k = rng.standard_normal((nk, n_kv * hd)).astype(np.float32)
    v = rng.standard_normal((nk, n_kv * hd)).astype(np.float32)
    q[3] *= 4.0  # a peaky row
    ref = np.zeros((T, n_heads * hd))
    kvm = n_heads // n_kv
    for h in range(n_heads):
        kh, vh = k[:, (h // kvm) * hd:(h // kvm + 1) * hd].astype(np.float64), v[:, (h // kvm) * hd:(h // kvm + 1) * hd].astype(np.float64)
        s = q[:, h * hd:(h + 1) * hd].astype(np.float64) @ kh.T / np.sqrt(hd)
        mask = np.arange(nk)[None, :] > (pos0 + np.arange(T))[:, None]
        s[mask] = -np.inf
        p = np.exp(s - s.max(axis=1, keepdims=True))
        ref[:, h * hd:(h + 1) * hd] = (p / p.sum(axis=1, keepdims=True)) @ vh
    out = T_mod.op_prefill_attention(q, k, v, pos0, n_heads, n_kv)
    err = float(np.abs(out - ref).max())
    print(f"prefill attention T={T} pos0={pos0} heads {n_heads}/{n_kv}: max err {err:.2e}")
    assert err <= 2e-5 * max(1.0, float(np.abs(ref).max()))
