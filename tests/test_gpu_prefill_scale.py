"""Batched prefill at the sizes it is run at: the persistent tcgen05 GEMM with many tiles per CTA, long and chunked prompts,
stale grow-only buffers, and a model wider than 4096.

k_gemm_q8 runs min(tiles, SMs) CTAs and each walks tile = blockIdx.x, + gridDim.x, ...  What carries from one tile to the
next -- the stage-ring count and its FULL / EMPTY parities, the accumulator-pair count (pair slot, TFULL / TEMPTY parities),
the scale-ring count, the epilogue's TMEM look-ahead into the next tile's first pair, the per-warp output patch -- only runs
when a CTA gets a second tile, i.e. when tiles > SMs.  The op-level shapes below are derived from the SM count (what the
launcher reads) so that every one of them does, in a different way.

The model-level part relies on every prefill kernel being independent per token row (norm / quantise: one block per token;
the GEMM: one thread folds one row in a fixed order; QK-norm / RoPE and the K / V split: per row; the attention kernel's key
tiles are aligned to absolute position 0 and a fully masked tile is a no-op: correction expf(0) = 1, P = 0).  So a prefix,
a chunked prompt, a rerun and a rerun after a longer prompt must all give BIT-identical cache rows and logits."""
import os

import numpy as np
import pytest

from oracle import binding as orc
from qwen3_rs_b200 import transformer as T_mod
from qwen3_rs_b200.sampler import argmax_last
from test_gpu_parity import check_layerwise, check_prefill_vs_oracle


def ref_gemm(xq, xs, wq, ws, gs):
    """out[t, r] = sum_g (f32(dot_g[t, r]) * ws[r, g]) * xs[t, g], groups folded left to right in float32 -- the oracle's matmul
    applied token by token.  The group dots are exact in float32: |dot| <= 128 * 127^2 < 2^24."""
    T, K = xq.shape
    N = wq.shape[0]
    ng = K // gs
    ws = ws.reshape(N, ng)
    acc = np.zeros((T, N), np.float32)
    for g in range(ng):
        d = xq[:, g * gs:(g + 1) * gs].astype(np.float32) @ wq[:, g * gs:(g + 1) * gs].astype(np.float32).T
        acc = acc + (d * ws[:, g]) * xs[:, g][:, None]
    return acc


def gemm_operands(T, N, K, gs, seed):
    rng = np.random.default_rng(seed)
    xq = rng.integers(-127, 128, size=(T, K), dtype=np.int8)
    xs = (rng.random((T, K // gs)) * 0.05 + 1e-3).astype(np.float32)
    wq = rng.integers(-127, 128, size=(N, K), dtype=np.int8)
    ws = (rng.random(N * K // gs) * 0.02 + 1e-4).astype(np.float32)
    xq[0, :] = 127   # extreme rows: |dot| reaches gs * 127^2
    wq[0, :] = -127
    return xq, xs, wq, ws


@pytest.mark.parametrize("T,N,K,gs", [(37, 256, 512, 64), (5, 128, 2432, 64), (3, 384, 4096, 128), (4, 128, 1024, 32)])
def test_numpy_gemm_reference_is_the_oracle_matmul(T, N, K, gs):
    """The reference the GEMM tests below rely on is bit-identical to the oracle's per-token matmul."""
    xq, xs, wq, ws = gemm_operands(T, N, K, gs, T + N + K)
    want = np.stack([orc.matmul(xq[t], xs[t], wq.reshape(-1), ws, K, N, gs) for t in range(T)])
    assert np.array_equal(ref_gemm(xq, xs, wq, ws, gs), want)


def num_sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def multi_tile_shapes(sms):
    """(T, N, K, gs, what) with tile t = m-tile t % mt, n-tile t / mt and grid = min(tiles, sms)."""
    return [
        # 1 pair / 1 K-stage per tile, ~8.6 tiles per CTA: the 4-stage ring and the 8-slot scale ring wrap inside one CTA's loop
        (1280, 128 * -(-86 * sms // 100), 128, 64, "K 128: 1 pair per tile, ~8.6 tiles per CTA"),
        # 19 pairs and 19 K-stages per tile (odd, not a multiple of 4; 4B down_proj at tp 4): the pair-slot parity flips from tile
        # to tile; the last m-tile has 44 rows
        (300, 128 * -(-(2 * sms + 7) // 3), 2432, 64, "K 2432: 19 pairs per tile, 2 SMs + 7 tiles"),
        (200, 128 * sms, 1024, 32, "K 1024 gs 32: exactly 2 tiles per CTA"),
        (77, 128 * (sms + 1), 256, 128, "K 256 gs 128: SMs + 1 tiles, one CTA runs a second tile"),
    ]


def check_gemm(T, N, K, gs, what):
    xq, xs, wq, ws = gemm_operands(T, N, K, gs, T + N + K)
    ref = ref_gemm(xq, xs, wq, ws, gs)
    tiles = (N // 128) * (-(-T // 128))
    out = T_mod.op_gemm_q8(xq, xs, wq, ws, T, N, K, gs, exact=True)
    bad = np.argwhere(~(out == ref))
    assert bad.size == 0, f"{what}: {len(bad)} outputs differ, first (t, n) {bad[:3].tolist()}, max err {float(np.nanmax(np.abs(out - ref)))}"
    # the drain q3_prefill runs: the same int32 group dots and group order, fused multiply-adds -> float round-off of the fold only
    fast = T_mod.op_gemm_q8(xq, xs, wq, ws, T, N, K, gs)
    scale = float(np.abs(ref).max())
    err = float(np.abs(fast - ref).max())
    print(f"GEMM T {T} N {N} K {K} gs {gs} ({tiles} tiles): exact mode bit-identical; fast drain max err {err:.2e} (|ref| max {scale:.1f})")
    assert np.isfinite(fast).all() and err <= 2e-6 * scale * np.sqrt(K / gs), what


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(4))
def test_gemm_many_tiles_per_cta_bit_identical(case):
    """Every CTA of the persistent GEMM runs more than one tile: exact mode bit-identical to the reference, the fast drain within
    the fold's round-off.  The output buffer is pre-filled with NaN and its padding rows are checked by q3_op_gemm_q8, so a
    skipped element or a stray store fails too."""
    sms = num_sms()
    T, N, K, gs, what = multi_tile_shapes(sms)[case]
    assert (N // 128) * (-(-T // 128)) > sms
    check_gemm(T, N, K, gs, what)


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("T,N,K,what", [(2048, 2 * 9728, 2560, "4B gate/up"), (2048, 2560, 9728, "4B down"),
                                        (2048, 2 * 12288, 4096, "8B gate/up"), (2048, 4096, 12288, "8B down")])
def test_gemm_real_prefill_shapes_bit_identical(T, N, K, what):
    """The bench's prefill GEMMs at T 2048, gs 64 (up to 21 tiles per CTA)."""
    check_gemm(T, N, K, 64, what)


# ---- model level: a 5120-wide model -------------------------------------------------------------
WIDE = ("wide", 64, 4)


def wide_model(ckpt):
    return T_mod.TransformerBuilder.new(ckpt(*WIDE)).build()


@pytest.fixture(scope="module")
def wide(ckpt):
    m = wide_model(ckpt)
    yield m
    m.close()


def run_prefill(m, toks, chunks=None):
    """reset, prefill `toks` (in one call, or as chunks [(a, b), ...] each at pos0 = a) -> (K / V rows of every layer, logits)."""
    m.reset()
    for a, b in chunks or [(0, len(toks))]:
        lg = m.prefill(toks[a:b], a)
    return [m.kv_read(l, 0, len(toks)) for l in range(m.get_config().n_layers)], lg


def assert_same_rows(got, want, n, label):
    for l, ((k, v), (kw, vw)) in enumerate(zip(got, want)):
        for name, a, b in (("K", k, kw), ("V", v, vw)):
            bad = np.nonzero(~(a[:n] == b[:n]).all(axis=1))[0]
            assert bad.size == 0, f"{label}: layer {l} {name} rows differ, first {bad[:5].tolist()} of {bad.size}, " \
                                  f"max err {float(np.abs(a[:n] - b[:n]).max()):.2e}"


def wide_tokens(n, seed=0):
    return np.random.default_rng(seed).integers(0, 4096, n).tolist()


@pytest.mark.gpu
def test_wide_prefill_prefix_chunk_and_rerun_invariance(wide):
    """2000 tokens (up to 6 GEMM tiles per CTA): the first 700 rows equal a 700-token prefill's; the chunks [0, 333),
    [333, 1201), [1201, 2000) at their pos0 (offsets that are no multiple of 32, 64 or 128) equal one prefill; a rerun is
    identical.  K / V rows of every layer and the last logits, bit for bit."""
    m = wide
    toks = wide_tokens(2000)
    full, lg = run_prefill(m, toks)
    assert np.isfinite(lg).all()
    again, lg2 = run_prefill(m, toks)
    assert_same_rows(again, full, 2000, "rerun")
    assert np.array_equal(lg2, lg), "rerun: logits differ"
    pre, _ = run_prefill(m, toks[:700])
    assert_same_rows(pre, full, 700, "700-token prefix")
    ch, lgc = run_prefill(m, toks, chunks=[(0, 333), (333, 1201), (1201, 2000)])
    assert_same_rows(ch, full, 2000, "chunks 333 / 868 / 799")
    assert np.array_equal(lgc, lg), f"chunks: logits differ by {float(np.abs(lgc - lg).max()):.2e}"


@pytest.mark.gpu
def test_wide_prefill_after_a_longer_one_is_unchanged(ckpt):
    """The prefill buffers only grow and are not cleared: after 2000 tokens their padding rows, and the K / V split buffer's
    rows past the prompt, hold the long prompt's data.  A 700-token prefill on a fresh handle, then 2000, then reset and
    700 again: the two 700-token results are identical."""
    m = wide_model(ckpt)
    try:
        toks = wide_tokens(2000, 1)
        first, lg1 = run_prefill(m, toks[:700])
        run_prefill(m, toks)
        last, lg2 = run_prefill(m, toks[:700])
        assert_same_rows(last, first, 700, "700 after 2000")
        assert np.array_equal(lg1, lg2)
    finally:
        m.close()


@pytest.mark.gpu
def test_wide_prefill_leaves_cache_rows_past_the_prompt_alone(wide):
    """Before prefilling 200 tokens at pos0 333, rows pos0 + T .. pos0 + Tpad + 127 of every layer hold a sentinel: afterwards
    they are untouched, and the prompt's rows equal those of one prefill of the whole 533 tokens (the attention reads no row
    past the causal horizon)."""
    m = wide
    c = m.get_config()
    kvd = c.n_kv_heads * c.head_dim
    toks = wide_tokens(533, 2)
    full, lg = run_prefill(m, toks)
    pos0, T = 333, 200
    lo, hi = pos0 + T, min(pos0 + 256 + 127, c.seq_len - 1)
    sentinel = np.full((hi + 1 - lo, kvd), -7777.25, np.float32)
    m.reset()
    m.prefill(toks[:pos0], 0)
    for l in range(c.n_layers):
        m.kv_write(l, lo, sentinel, sentinel)
    lg2 = m.prefill(toks[pos0:], pos0)
    for l in range(c.n_layers):
        k, v = m.kv_read(l, lo, hi + 1 - lo)
        assert np.array_equal(k, sentinel) and np.array_equal(v, sentinel), f"layer {l}: rows past the prompt were written"
    assert_same_rows([m.kv_read(l, 0, lo) for l in range(c.n_layers)], full, lo, "with sentinel rows")
    assert np.array_equal(lg2, lg)


@pytest.mark.gpu
def test_wide_prefill_matches_oracle(wide, ckpt):
    """640 tokens through q3_prefill (every GEMM has more tiles than SMs, the dim > 4096 norm kernel) against the oracle's
    640 sequential forwards."""
    orc.set_threads(os.cpu_count() or 1)
    check_prefill_vs_oracle(wide, ckpt(*WIDE), wide_tokens(640, 3), "wide gs64")


@pytest.mark.gpu
def test_wide_decode_graph_path_exact_mode_and_layerwise(wide, ckpt):
    """At dim 5120 the persistent decode kernel declines the shape, so the CUDA-graph path is the default decode path: exact
    mode reproduces the oracle's logits (8 greedy tokens, 1e-6), and fast mode passes the layer-wise comparison."""
    m = wide
    with pytest.raises(T_mod.Q3Error):
        m.set_decode_path(1)
    path = ckpt(*WIDE)
    o = orc.Model(path)
    try:
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
        finally:
            m.set_exact(False)
        print(f"wide exact mode: 8 greedy tokens identical, max |dlogit| {worst:.2e}")
        assert worst <= 1e-6
        check_layerwise(m, o, orc.Model(path), [1, 3001, 17, 99], "wide")
    finally:
        o.close()
