"""q3_score: per-position log-probabilities and greedy argmax of a token sequence in one batched pass.

The reduction (k_logprobs) is checked on its own against float64; exact mode against the committed golden logits (there the
logits are the reference's bit for bit, so the scores are the reduction of the reference's own logits); the batched fast path
against the oracle's sequential forwards with the oracle's own re-association noise as the yardstick.  The fast path's rows
are independent (per-row norm / quantise, one GEMM row folded by one thread in a fixed order, one CTA per reduced row), so a
prefix, a split into two calls, a rerun and the KV cache it leaves must all be bit-identical to the corresponding prefill."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN_CASES
from oracle import binding as orc
from qwen3_rs_b200 import generation
from qwen3_rs_b200 import transformer as T
from qwen3_rs_b200.sampler import argmax_last
from test_gpu_tp import _free_port, _ngpu

pytestmark = pytest.mark.gpu


def lsm64(lg):
    """float64 log-softmax along the last axis."""
    x = np.asarray(lg, np.float64)
    m = x.max(axis=-1, keepdims=True)
    return x - m - np.log(np.exp(x - m).sum(axis=-1, keepdims=True))


def lp_bound(lp64):
    return 4e-6 * (1.0 + np.abs(lp64))


# ---- the reduction alone ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,n", [(1, 256), (37, 768), (5, 4096), (3, 151936)])
@pytest.mark.parametrize("scale", [1.0, 30.0])
@pytest.mark.parametrize("offset", [0.0, 1e4, -1e4])
def test_op_logprobs_against_float64(rows, n, scale, offset):
    rng = np.random.default_rng(rows * 7 + n + int(scale))
    lg = (rng.standard_normal((rows, n)) * scale + offset).astype(np.float32)
    ref = lsm64(lg)
    worst = 0.0
    for targets in (lg.argmax(axis=1), lg.argmin(axis=1), rng.integers(0, n, rows)):
        lp, am = T.op_logprobs(lg, targets)
        want = ref[np.arange(rows), targets]
        err = np.abs(lp.astype(np.float64) - want)
        worst = max(worst, float((err / (1.0 + np.abs(want))).max()))
        assert (err <= lp_bound(want)).all(), (float(err.max()), targets)
        assert am.tolist() == [argmax_last(r) for r in lg]
        lp2, am2 = T.op_logprobs(lg, targets)  # a rerun: the same bits
        assert np.array_equal(lp2.view(np.uint32), lp.view(np.uint32)) and np.array_equal(am2, am)
        if rows > 1:  # one row launched alone: the same bits as inside the batch
            lp1, am1 = T.op_logprobs(lg[rows - 1:], targets[rows - 1:])
            assert lp1.view(np.uint32)[0] == lp.view(np.uint32)[-1] and am1[0] == am[-1]
    print(f"op_logprobs rows {rows} n {n} scale {scale} offset {offset}: worst |dlp| / (1 + |lp|) {worst:.2e}")


@pytest.mark.parametrize("n", [256, 768, 151936])
def test_op_logprobs_ties_and_an_all_equal_row(n):
    rng = np.random.default_rng(n)
    lg = rng.standard_normal((3, n)).astype(np.float32)
    lg[0] = 0.25                                    # all equal: lp = -log n at any target, argmax = n - 1
    top = float(lg[1].max()) + 1.0
    for i in (3, 100, n // 2, n - 7):               # planted ties for the maximum: the last one wins
        lg[1, i] = top
    lg[2, :] = -5.0
    lg[2, [0, 1, n // 3]] = 2.0                     # ties at the front of the row
    targets = np.array([n // 2, n - 7, 1], np.int32)
    lp, am = T.op_logprobs(lg, targets)
    assert am.tolist() == [n - 1, n - 7, n // 3]
    want = lsm64(lg)[np.arange(3), targets]
    assert abs(float(lp[0]) + np.log(n)) <= 4e-6 * (1 + np.log(n))
    assert (np.abs(lp - want) <= lp_bound(want)).all()
    _, am_only = T.op_logprobs(lg, None)            # argmax alone needs no targets
    assert np.array_equal(am_only, am)


def test_op_logprobs_argument_errors_write_nothing():
    lg = np.zeros((2, 256), np.float32)
    lp = np.full(2, -7.5, np.float32)
    am = np.full(2, -3, np.int32)
    L = T.load_library()
    p = T._ptr
    for rows, n, tg, lpo, amo in ((2, 256, np.array([0, 256], np.int32), lp, am),     # target out of range
                                  (2, 256, np.array([0, -1], np.int32), lp, am),
                                  (2, 256, None, lp, am),                             # logprobs without targets
                                  (2, 256, np.array([0, 1], np.int32), None, None),   # no output
                                  (0, 256, np.array([0, 1], np.int32), lp, am),
                                  (2, 0, np.array([0, 1], np.int32), lp, am)):
        assert L.q3_op_logprobs(0, p(lg), rows, n, p(tg), p(lpo), p(amo)) == -1
        assert (lp == -7.5).all() and (am == -3).all()


# ---- models -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def models(ckpt):
    cache = {}

    def get(name, gs, seed):
        key = (name, gs, seed)
        if key not in cache:
            cache[key] = T.TransformerBuilder.new(ckpt(name, gs, seed)).build()
        return cache[key]

    yield get
    for m in cache.values():
        m.close()


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_exact_mode_scores_the_golden_logits(models, golden, name, gs, seed):
    """Exact mode: the golden sequence (prompt + greedy) scored with targets = the next token.  Where golden logits exist (the
    teacher-forced logits of the whole sequence), the argmax is theirs and the log-probabilities are their float64
    log-softmax within the operator bound; perplexity over those positions to 1e-5 relative.  The golden greedy tokens come
    from the reference's generate(), which never forwards the prompt tokens before the last one (generation.rs:26-28, their
    cache rows stay zero): scored the same way -- from pos0 = len(prompt) - 1 on a reset cache -- the argmax is the next greedy
    token at every position."""
    key = f"{name}_gs{gs}"
    m = models(name, gs, seed)
    prompt, greedy = golden[key + "_prompt"].tolist(), golden[key + "_greedy"].tolist()
    seq = prompt + greedy
    lg = golden[key + "_logits"]
    p0 = len(prompt) - 1
    m.set_exact(True)
    try:
        m.reset()
        _, am_gen = m.score(seq[p0:-1], pos0=p0)
        m.reset()
        lp, am = m.score(seq[:-1], targets=seq[1:])
        npos = lg.shape[0]
        ppl, total = generation.perplexity(m, seq[:npos + 1])
    finally:
        m.set_exact(False)
    assert am_gen.tolist() == greedy
    want = lsm64(lg)[np.arange(npos), seq[1:npos + 1]]
    assert [int(a) for a in am[:npos]] == [argmax_last(r) for r in lg]
    err = np.abs(lp[:npos].astype(np.float64) - want)
    print(f"{key} exact mode: {len(seq) - 1} positions scored, worst |dlp| vs golden float64 {err.max():.2e}")
    assert (err <= lp_bound(want)).all()
    assert abs(ppl - np.exp(-want.mean())) <= 1e-5 * np.exp(-want.mean())
    assert abs(total - want.sum()) <= 1e-5 * max(1.0, abs(want.sum()))


def oracle_logits(path, toks, perturb):
    o = orc.Model(path)
    try:
        orc.set_perturb(perturb)
        return np.stack([o.forward(t, p) for p, t in enumerate(toks)])
    finally:
        orc.set_perturb(0)
        o.close()


def check_scores_vs_oracle(lp, am, lo, lo2, targets, label):
    """Fast-path scores (lp, am) against the oracle's logits lo, with the perturbed oracle's lo2 as the noise yardstick."""
    idx = np.arange(len(targets))
    ref, noise = lsm64(lo)[idx, targets], lsm64(lo2)[idx, targets]
    d = np.abs(lp.astype(np.float64) - ref)
    dn = np.abs(noise - ref)
    bound = 2 * (0.05 * float(np.abs(lo).max()) + 1e-2)
    print(f"{label}: max |dlp| {d.max():.2e} (bound {bound:.2e}), median {np.median(d):.2e} (oracle re-association: "
          f"max {dn.max():.2e}, median {np.median(dn):.2e})")
    assert d.max() <= bound
    assert np.median(d) <= max(1e-5, 3 * np.median(dn))
    lsm = lsm64(lo)
    for p in idx:
        top2 = np.sort(lo[p])[-2:]
        if top2[1] - top2[0] > 0.5:
            assert am[p] == argmax_last(lo[p]), (label, p)
        else:  # a near tie: the chosen token is as likely as the best within the bound
            assert lsm[p].max() - lsm[p, am[p]] <= bound, (label, p)


FAST_CASES = [("tiny-untied", 64, 1, 37), ("small", 128, 2, 130), ("small", 64, 3, 200)]


@pytest.mark.parametrize("name,gs,seed,n", FAST_CASES)
def test_fast_path_scores_match_oracle(models, ckpt, name, gs, seed, n):
    m = models(name, gs, seed)
    toks = np.random.default_rng(n + 11).integers(0, m.get_config().vocab_size, n + 1).tolist()
    targets = toks[1:]
    path = ckpt(name, gs, seed)
    lo, lo2 = oracle_logits(path, toks[:n], 0), oracle_logits(path, toks[:n], 1)
    m.reset()
    lp, am = m.score(toks[:n], targets=targets)
    check_scores_vs_oracle(lp, am, lo, lo2, np.array(targets), f"{name} gs{gs} T {n}")


WIDE = ("wide", 64, 4)


def wide_tokens(n, seed):
    return np.random.default_rng(seed).integers(0, 4096, n).tolist()


def test_wide_fast_path_scores_match_oracle(models, ckpt):
    """dim 5120 (the > 4096 norm kernel) at T 640: two lm_head row chunks."""
    orc.set_threads(os.cpu_count() or 1)
    m = models(*WIDE)
    toks = wide_tokens(641, 3)
    path = ckpt(*WIDE)
    lo, lo2 = oracle_logits(path, toks[:640], 0), oracle_logits(path, toks[:640], 1)
    m.reset()
    lp, am = m.score(toks[:640], targets=toks[1:])
    check_scores_vs_oracle(lp, am, lo, lo2, np.array(toks[1:]), "wide gs64 T 640")


def bits(a):
    return np.asarray(a).view(np.uint32)


def kv_rows(m, n):
    return [m.kv_read(l, 0, n) for l in range(m.get_config().n_layers)]


@pytest.mark.parametrize("name,gs,seed,n,splits", [("small", 64, 3, 500, (333,)), ("wide", 64, 4, 2000, (333, 700))])
def test_fast_path_bit_identity(models, name, gs, seed, n, splits):
    """Rerun, prefix (including n 1), split into two calls at pos0 > 0, the KV cache it leaves, and the decode step after it:
    all bit-identical to the full call / to q3_prefill.  At 2000 tokens the lm_head runs 4 row chunks, the last one ragged."""
    m = models(name, gs, seed)
    c = m.get_config()
    toks = np.random.default_rng(n).integers(0, c.vocab_size, n + 1).tolist()
    t, tg = toks[:n], toks[1:]
    m.reset()
    lp, am = m.score(t, targets=tg)
    assert np.isfinite(lp).all() and (lp <= 0).all()
    kv_score = kv_rows(m, c.seq_len if c.seq_len <= n + 256 else n + 256)
    nxt_score = m.forward(toks[n], n)
    m.reset()
    lp2, am2 = m.score(t, targets=tg)
    assert np.array_equal(bits(lp2), bits(lp)) and np.array_equal(am2, am), "rerun"
    for k in (1, 129, 333, n - 1):
        m.reset()
        lpk, amk = m.score(t[:k], targets=tg[:k])
        assert np.array_equal(bits(lpk), bits(lp[:k])) and np.array_equal(amk, am[:k]), f"prefix {k}"
    _, am_only = m.score(t, want_argmax=True)
    assert np.array_equal(am_only, am), "argmax without log-probabilities"
    for a in splits:
        m.reset()
        lpa, ama = m.score(t[:a], targets=tg[:a])  # the last target is t[a], scored at position a - 1
        lpb, amb = m.score(t[a:], targets=tg[a:], pos0=a)
        assert np.array_equal(bits(np.concatenate([lpa, lpb])), bits(lp)), f"split at {a}"
        assert np.array_equal(np.concatenate([ama, amb]), am), f"split at {a}"
    # the cache and the next decode step: as after q3_prefill of the same tokens
    m.reset()
    m.prefill(t, 0, want_logits=False)
    kv_pf = kv_rows(m, len(kv_score[0][0]))
    nxt_pf = m.forward(toks[n], n)
    for l, ((k, v), (kp, vp)) in enumerate(zip(kv_score, kv_pf)):
        assert np.array_equal(k, kp) and np.array_equal(v, vp), f"layer {l}: KV rows differ from q3_prefill's"
        assert not k[n:].any() and not v[n:].any(), f"layer {l}: rows past the prompt written"
    assert np.array_equal(bits(nxt_score), bits(nxt_pf)), "decode after q3_score differs from decode after q3_prefill"


def test_score_argument_errors_write_nothing(models):
    m = models("small", 64, 3)
    c = m.get_config()
    L = T.load_library()
    p = T._ptr
    toks = np.arange(1, 9, dtype=np.int32)
    tg = np.arange(2, 10, dtype=np.int32)
    lp = np.full(8, -7.5, np.float32)
    am = np.full(8, -3, np.int32)
    bad_tok = toks.copy()
    bad_tok[5] = c.vocab_size
    bad_tg = tg.copy()
    bad_tg[7] = -1
    cases = [(toks, 0, 0, tg, lp, am), (toks, 8, c.seq_len - 7, tg, lp, am), (toks, 8, -1, tg, lp, am),
             (bad_tok, 8, 0, tg, lp, am), (toks, 8, 0, bad_tg, lp, am), (toks, 8, 0, None, lp, am), (toks, 8, 0, tg, None, None)]
    for tk, n, pos0, tgt, lpo, amo in cases:
        assert L.q3_score(C.c_void_p(m._h), p(tk), n, pos0, p(tgt), p(lpo), p(amo)) == -1
        assert (lp == -7.5).all() and (am == -3).all()
    m.reset()
    lp_ok, am_ok = m.score(toks.tolist(), targets=tg.tolist())  # the handle stays usable
    assert np.isfinite(lp_ok).all()
    with pytest.raises(ValueError):
        generation.perplexity(m, list(range(c.seq_len + 2)))


# ---- tensor parallel ----------------------------------------------------------------------------------------------------
def _tp_worker(rank, world, port, path, n, q):
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        m = T.TransformerBuilder.new(path).with_device(rank).with_tensor_parallel(rank, world).build()
        T.tp_connect(m, dist)
        toks = np.random.default_rng(n).integers(0, m.get_config().vocab_size, n + 1).tolist()
        lp, am = m.score(toks[:n], targets=toks[1:])
        code = 0
        try:
            m.set_exact(True)
            m.score(toks[:n], targets=toks[1:])
        except T.Q3Error as e:
            code = e.code
        q.put((rank, {"lp": lp, "am": am, "toks": toks, "exact_code": code}))
        dist.barrier()
        m.close()
    except Exception as e:  # noqa: BLE001 -- surface the failure to the parent instead of a queue timeout
        import traceback

        q.put((rank, {"error": repr(e) + "\n" + traceback.format_exc()}))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("name,gs,seed,world", [("small", 64, 3, 2), ("small8", 64, 5, 4)])
def test_tensor_parallel_scores(ckpt, name, gs, seed, world):
    """Every rank runs the full lm_head on the all-reduced residual stream: the ranks' results are bit-identical and match the
    oracle as on one GPU.  Exact mode is single-GPU: Q3_EUNSUPPORTED."""
    import torch.multiprocessing as mp

    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    path, n = ckpt(name, gs, seed), 120
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_tp_worker, args=(r, world, port, path, n, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    got = dict(q.get(timeout=240) for _ in range(world))
    for pr in procs:
        pr.join(60)
    for r in range(world):
        assert "error" not in got[r], got[r]["error"]
        assert got[r]["exact_code"] == -5
    for r in range(1, world):
        assert np.array_equal(bits(got[r]["lp"]), bits(got[0]["lp"])) and np.array_equal(got[r]["am"], got[0]["am"])
    toks = got[0]["toks"]
    lo, lo2 = oracle_logits(path, toks[:n], 0), oracle_logits(path, toks[:n], 1)
    check_scores_vs_oracle(got[0]["lp"], got[0]["am"], lo, lo2, np.array(toks[1:]), f"{name} gs{gs} tp{world}")
