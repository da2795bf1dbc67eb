"""q3_forward_multi and q3_decode_speculative.

forward_multi runs n <= 8 decode steps of consecutive positions in one pass over the weights; each token's row (logits, argmax,
K/V cache row) must be bit-identical to the single-token step of the multi-kernel (graph) path.  decode_speculative builds
greedy decoding on it, so its tokens and the target's cache must be exactly decode_greedy's on the graph path whatever the
draft proposes.  Shapes: one per group size and GQA factor (1, 2, 4, 8), all with a 1024-token vocabulary so that any of them
can draft for another; K/V caches are filled with seeded random rows (q3_kv_write) so that long contexts cost no decode steps."""
import ctypes as C
import os
import shutil

import numpy as np
import pytest

from conftest import GOLDEN_CASES
from qwen3_rs_b200 import synth
from qwen3_rs_b200 import transformer as T
from qwen3_rs_b200.sampler import argmax_last

pytestmark = pytest.mark.gpu

V = 1024
SHAPES = {
    "g1": synth.Shape("g1", 256, 768, 2, 2, 2, vocab_size=V, max_seq_len=4096, tied=False),
    "g2": synth.Shape("g2", 256, 512, 3, 4, 2, vocab_size=V, max_seq_len=512, tied=True),
    "g4": synth.Shape("g4", 512, 1024, 2, 8, 2, vocab_size=V, max_seq_len=512, tied=False),
    "g8": synth.Shape("g8", 256, 512, 2, 8, 1, vocab_size=V, max_seq_len=512, tied=False),
    "d-small": synth.Shape("d-small", 128, 384, 1, 1, 1, vocab_size=V, max_seq_len=512, tied=True),
    # down_proj K = 57344 at gs 32: 64512 staged bytes per token, so at most 3 tokens fit a GEMV's 227 KB of shared memory and
    # the multi-token step splits its tokens into groups (n 4 = 3 + 1, n 8 = 3 + 3 + 2)
    "wide-ffn": synth.Shape("wide-ffn", 128, 57344, 1, 1, 1, vocab_size=V, max_seq_len=64, tied=True),
}
CASES = [("g1", 32), ("g2", 64), ("g4", 128), ("g8", 64)]  # (shape, group size): GQA 1, 2, 4, 8
SENTINEL = np.float32(-1234.5)
EINVAL, EUNSUPPORTED = -1, -5  # Q3_EINVAL, Q3_EUNSUPPORTED


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def handle(tmp_path_factory):
    """handle(shape, gs, seed, tag) -> a Transformer (cached per tag, so two tags give two handles on one checkpoint);
    handle.path(shape, gs, seed) -> the exported checkpoint."""
    d = str(tmp_path_factory.mktemp("spec"))
    paths, cache = {}, {}

    def path(name, gs, seed=0):
        if (name, gs, seed) not in paths:
            p = os.path.join(d, f"{name}_gs{gs}_s{seed}.bin")
            synth.export_synthetic(SHAPES[name], p, gs, seed=seed)
            paths[(name, gs, seed)] = p
        return paths[(name, gs, seed)]

    def get(name, gs, seed=0, tag=""):
        key = (name, gs, seed, tag)
        if key not in cache:
            cache[key] = T.TransformerBuilder.new(path(name, gs, seed)).build()
        return cache[key]

    get.path = path
    yield get
    for m in cache.values():
        m.close()
    shutil.rmtree(d, ignore_errors=True)


def fill_cache(ms, rows, seed, scale=0.5):
    """The same seeded random K/V rows [0, rows) in every handle of ms (one shape)."""
    cfg = ms[0].get_config()
    kv = cfg.n_kv_heads * cfg.head_dim
    rng = np.random.default_rng(seed)
    for l in range(cfg.n_layers):
        k = (rng.standard_normal((rows, kv)) * scale).astype(np.float32)
        v = (rng.standard_normal((rows, kv)) * scale).astype(np.float32)
        for m in ms:
            if rows:
                m.kv_write(l, 0, k, v)


def kv_block(m, pos0, n):
    return [m.kv_read(l, pos0, n) for l in range(m.get_config().n_layers)]


def assert_kv_equal(a, b, label):
    for l, ((ka, va), (kb, vb)) in enumerate(zip(a, b)):
        assert np.array_equal(bits(ka), bits(kb)) and np.array_equal(bits(va), bits(vb)), f"{label}: layer {l} K/V differ"


def write_sentinel(m, pos0, n):
    cfg = m.get_config()
    kv = cfg.n_kv_heads * cfg.head_dim
    s = np.full((n, kv), SENTINEL, np.float32)
    for l in range(cfg.n_layers):
        m.kv_write(l, pos0, s, s)


def assert_sentinel(m, pos0, n, label):
    for l, (k, v) in enumerate(kv_block(m, pos0, n)):
        assert (k == SENTINEL).all() and (v == SENTINEL).all(), f"{label}: layer {l} row >= {pos0} was written"


# ---- 1. row bit-identity ---------------------------------------------------------------------------------------------------
def check_rows(m, ref, pos0, seed, label):
    """forward_multi at pos0 for n = 1 .. 8 against n graph-path forwards on ref (same cache rows)."""
    rng = np.random.default_rng(seed)
    for n in range(1, T.MULTI_MAX + 1):
        toks = rng.integers(0, V, n).tolist()
        am, lg = m.forward_multi(toks, pos0, want_logits=True)
        want = np.stack([ref.forward(t, pos0 + i) for i, t in enumerate(toks)])
        bad = np.argwhere(bits(lg) != bits(want))
        assert bad.size == 0, f"{label} pos0 {pos0} n {n}: logits differ at {bad[:4].tolist()}"
        assert am.tolist() == [argmax_last(r) for r in want], f"{label} pos0 {pos0} n {n}: argmax"
        assert_kv_equal(kv_block(m, pos0, n), kv_block(ref, pos0, n), f"{label} pos0 {pos0} n {n}")


@pytest.mark.parametrize("name,gs", CASES)
def test_forward_multi_rows_bit_identical(handle, name, gs):
    """Every n in 1..8 at pos0 0, on both sides of a split-count change (ATTN_MIN_CHUNK = 128) and, on the long-context shape,
    at a few thousand cached rows and against the end of the context.  The multi handle stays on its default path (the
    persistent kernel where available): forward_multi does not depend on it."""
    m, ref = handle(name, gs, 0, "a"), handle(name, gs, 0, "b")
    ref.set_decode_path(0)
    seq = m.get_config().seq_len
    positions = [0, 121, 125, 127, 128, 129, 133, 250, 256]
    if seq >= 4096:
        positions += [3000, 4088]
    fill_cache([m, ref], max(positions) + 8, seed=gs)
    for p in positions:
        check_rows(m, ref, p, p + gs, name)


def test_forward_multi_rows_bit_identical_when_tokens_go_in_groups(handle):
    m, ref = handle("wide-ffn", 32, 0, "a"), handle("wide-ffn", 32, 0, "b")
    ref.set_decode_path(0)
    fill_cache([m, ref], 40, seed=3)
    for p in (0, 29):
        check_rows(m, ref, p, p, "wide-ffn")


@pytest.mark.parametrize("mask", [31, 8])
def test_forward_multi_exact_mode_runs_the_exact_steps(handle, mask):
    """Exact mode (all bits) and a partial mask (attention only): the n single-token steps of that mode."""
    m, ref = handle("g2", 64, 0, "a"), handle("g2", 64, 0, "b")
    ref.set_decode_path(0)
    fill_cache([m, ref], 140, seed=mask)
    m.set_exact_mask(mask)
    ref.set_exact_mask(mask)
    try:
        for p in (0, 126):
            check_rows(m, ref, p, p + mask, f"exact mask {mask}")
    finally:
        m.set_exact_mask(0)
        ref.set_exact_mask(0)


def test_forward_multi_without_logits_and_repeated(handle):
    """Argmax only, and the same call twice (the graph of each n is captured once and replayed)."""
    m, ref = handle("g4", 128, 0, "a"), handle("g4", 128, 0, "b")
    ref.set_decode_path(0)
    fill_cache([m, ref], 64, seed=5)
    toks = [3, 1, 4, 1, 5, 9, 2]
    a1, lg = m.forward_multi(toks, 40)
    a2, _ = m.forward_multi(toks, 40)
    assert lg is None and a1.tolist() == a2.tolist()
    assert a1.tolist() == [ref.forward_argmax(t, 40 + i) for i, t in enumerate(toks)]


# ---- 2. speculative = greedy -------------------------------------------------------------------------------------------------
DRAFTS = ["same-graph", "same-persistent", "other-seed", "smaller-shape", "reset-cache"]


def make_draft(handle, name, gs, kind, rows):
    if kind in ("same-graph", "same-persistent", "reset-cache"):
        d = handle(name, gs, 0, "draft")
        d.set_decode_path(0)
        if kind == "same-persistent":
            try:
                d.set_decode_path(1)
            except T.Q3Error:
                pytest.skip("no persistent kernel for this shape")
        if kind == "reset-cache":
            d.reset()
        else:
            fill_cache([d], rows, seed=11)
        return d
    d = handle(name, gs, 1, "draft") if kind == "other-seed" else handle("d-small", 64, 3, "draft")
    d.set_decode_path(0)
    fill_cache([d], rows, seed=13)
    return d


@pytest.mark.parametrize("name,gs", CASES)
@pytest.mark.parametrize("k", [1, 3, 7])
@pytest.mark.parametrize("kind", DRAFTS)
def test_speculative_equals_greedy(handle, name, gs, k, kind):
    pos0, n, first = 100, 48, 7
    tgt, ref = handle(name, gs, 0, "a"), handle(name, gs, 0, "b")
    ref.set_decode_path(0)
    draft = make_draft(handle, name, gs, kind, pos0)
    fill_cache([tgt, ref], pos0, seed=11)  # the same-checkpoint drafts hold these rows too
    for m in (tgt, ref):
        write_sentinel(m, pos0, n + 16)
    want = ref.decode_greedy(first, pos0, n)
    got, st = tgt.decode_speculative(draft, first, pos0, n, k)
    assert got == want, (kind, k, got, want)
    assert_kv_equal(kv_block(tgt, 0, pos0 + n), kv_block(ref, 0, pos0 + n), f"{kind} k {k}")
    assert_sentinel(tgt, pos0 + n, 16, f"{kind} k {k}")
    assert st["accepted"] <= st["drafted"] and st["rounds"] + st["accepted"] == n, st
    if kind == "same-graph":
        assert st["accepted"] == st["drafted"], st
    print(f"{name} gs{gs} k {k} {kind}: {st}")


# ---- 3. reference parity -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden_models(ckpt):
    cache = {}

    def get(name, gs, seed, tag):
        if (name, gs, seed, tag) not in cache:
            cache[(name, gs, seed, tag)] = T.TransformerBuilder.new(ckpt(name, gs, seed)).build()
        return cache[(name, gs, seed, tag)]

    yield get
    for m in cache.values():
        m.close()


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_speculative_exact_mode_gives_the_oracle_greedy_tokens(golden_models, golden, name, gs, seed):
    key = f"{name}_gs{gs}"
    prompt, want = golden[key + "_prompt"].tolist(), golden[key + "_greedy"].tolist()
    tgt, draft = golden_models(name, gs, seed, "t"), golden_models(name, gs, seed, "d")
    tgt.set_exact(True)
    try:
        for m in (tgt, draft):  # the reference's generate never forwards the prompt tokens before the last (generate_fast)
            m.reset()
        got, st = tgt.decode_speculative(draft, prompt[-1], len(prompt) - 1, len(want), 3)
        assert got == want, st
    finally:
        tgt.set_exact(False)


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_speculative_fast_mode_vs_persistent_greedy(golden_models, golden, name, gs, seed):
    """The default (persistent) path's greedy tokens agree with the speculative ones up to the first position whose top-2
    margin on the graph path is inside the fast-mode noise (the paths reduce in different orders)."""
    key = f"{name}_gs{gs}"
    prompt, n = golden[key + "_prompt"].tolist(), len(golden[key + "_greedy"])
    tgt, draft = golden_models(name, gs, seed, "t"), golden_models(name, gs, seed, "d")
    for m in (tgt, draft):
        m.reset()
    got, _ = tgt.decode_speculative(draft, prompt[-1], len(prompt) - 1, n, 7)
    tgt.reset()
    fast = tgt.decode_greedy(prompt[-1], len(prompt) - 1, n)
    if fast != got:
        p = next(i for i in range(n) if fast[i] != got[i])
        seq = [prompt[-1]] + got
        persistent = tgt.launches_per_step == 1
        tgt.set_decode_path(0)
        try:  # the cache holds the persistent path's rows of the common prefix: a margin within the noise of the graph path's
            lg = tgt.forward(seq[p], len(prompt) - 1 + p)
        finally:
            tgt.set_decode_path(1 if persistent else 0)
        top2 = np.sort(lg)[-2:]
        assert top2[1] - top2[0] < 2e-2, (p, float(top2[1] - top2[0]))


# ---- 4. edges and errors -----------------------------------------------------------------------------------------------------
def test_speculative_edges(handle):
    tgt, ref = handle("g2", 64, 0, "a"), handle("g2", 64, 0, "b")
    draft = handle("g2", 64, 1, "draft")
    ref.set_decode_path(0)
    seq = tgt.get_config().seq_len
    for pos0, n, k in [(20, 0, 3), (20, 1, 3), (20, 3, 7), (seq - 10, 10, 7), (seq - 1, 1, 1)]:
        fill_cache([tgt, ref], pos0, seed=pos0)
        fill_cache([draft], pos0, seed=pos0 + 1)
        tail = min(16, seq - pos0 - n)
        for m in (tgt, ref):
            write_sentinel(m, pos0, n + tail)
        got, st = tgt.decode_speculative(draft, 5, pos0, n, k)
        want = ref.decode_greedy(5, pos0, n) if n else []
        assert got == want, (pos0, n, k)
        assert_kv_equal(kv_block(tgt, 0, pos0 + n), kv_block(ref, 0, pos0 + n), f"pos0 {pos0} n {n} k {k}")
        if tail:
            assert_sentinel(tgt, pos0 + n, tail, f"pos0 {pos0} n {n} k {k}")
        assert st["rounds"] + st["accepted"] == n and st["drafted"] <= n * k


def test_invalid_arguments_are_errors_that_write_nothing(handle, golden_models):
    L = T.load_library()
    tgt, draft = handle("g2", 64, 0, "a"), handle("g2", 64, 1, "draft")
    other_vocab = golden_models("micro", 32, 7, "v")  # vocab 256
    seq = tgt.get_config().seq_len
    fill_cache([tgt], 32, seed=1)
    write_sentinel(tgt, 32, 16)

    def spec(t, d, first, pos0, n, k):
        out = np.full(max(n, 1) + 4, -7, np.int32)
        st = [C.c_int(-3) for _ in range(3)]
        rc = L.q3_decode_speculative(t._h, d._h, first, pos0, n, k, out.ctypes.data_as(C.c_void_p), *[C.byref(x) for x in st])
        assert (out == -7).all() and all(x.value == -3 for x in st)
        return rc

    for args in [(tgt, tgt, 5, 32, 4, 3), (tgt, other_vocab, 5, 32, 4, 3), (tgt, draft, 5, 32, 4, 0), (tgt, draft, 5, 32, 4, T.MULTI_MAX),
                 (tgt, draft, -1, 32, 4, 3), (tgt, draft, V, 32, 4, 3), (tgt, draft, 5, -1, 4, 3), (tgt, draft, 5, seq - 3, 4, 3),
                 (tgt, draft, 5, 32, -1, 3)]:
        assert spec(*args) == EINVAL, args
    am = np.full(T.MULTI_MAX + 2, -7, np.int32)
    for toks, pos0 in [(list(range(T.MULTI_MAX + 1)), 32), ([], 32), ([1, V], 32), ([1, -1], 32), ([1, 2], -1), ([1, 2], seq - 1)]:
        t = np.asarray(toks + [0], np.int32)
        rc = L.q3_forward_multi(tgt._h, t.ctypes.data_as(C.c_void_p), len(toks), pos0, am.ctypes.data_as(C.c_void_p), None)
        assert rc == EINVAL and (am == -7).all(), (toks, pos0)
    t = np.asarray([1, 2], np.int32)
    assert L.q3_forward_multi(tgt._h, t.ctypes.data_as(C.c_void_p), 2, 32, None, None) == EINVAL
    assert L.q3_forward_multi(tgt._h, None, 2, 32, am.ctypes.data_as(C.c_void_p), None) == EINVAL
    assert_sentinel(tgt, 32, 16, "invalid arguments")
    with pytest.raises(ValueError):
        tgt.forward_multi(list(range(T.MULTI_MAX + 1)), 0)
    with pytest.raises(ValueError):
        tgt.decode_speculative(draft, 5, 32, 4, T.MULTI_MAX)


def test_draft_on_another_device_is_refused(handle):
    tgt = handle("g2", 64, 0, "a")
    try:
        other = T.TransformerBuilder.new(handle.path("g2", 64, 1)).with_device(1).build()
    except T.Q3Error as e:
        pytest.skip(f"no second device: {e}")
    try:
        with pytest.raises(T.Q3Error) as e:
            tgt.decode_speculative(other, 5, 0, 4, 3)
        assert e.value.code == EINVAL
    finally:
        other.close()


def test_tensor_parallel_handle_is_unsupported(ckpt):
    try:
        m = T.TransformerBuilder.new(ckpt("small8", 64, 0)).with_tensor_parallel(0, 2).build()
    except T.Q3Error as e:
        pytest.skip(f"no tensor-parallel handle here: {e}")
    try:
        other = T.TransformerBuilder.new(ckpt("small8", 64, 0)).build()
        try:
            with pytest.raises(T.Q3Error) as e:
                m.forward_multi([1, 2], 0)
            assert e.value.code == EUNSUPPORTED
            with pytest.raises(T.Q3Error) as e:
                m.decode_speculative(other, 1, 0, 4, 3)
            assert e.value.code == EUNSUPPORTED
            with pytest.raises(T.Q3Error) as e:
                other.decode_speculative(m, 1, 0, 4, 3)
            assert e.value.code == EUNSUPPORTED
        finally:
            other.close()
    finally:
        m.close()
