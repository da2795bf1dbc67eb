"""q3_score_topk: the k most likely tokens and their log-probabilities at every position, in one batched pass.

The selection (k_topk_logprobs) is checked on its own against float64 log-softmax and a stable sort by (value descending,
index descending), on rows chosen to reach every branch of the radix select: random rows (first gather), ±1e4 offsets and
values a few ulps apart (refinement digits), all-equal rows (down into the index bits), ties straddling the k-th place and
rows containing -inf.  Through the engine its extra outputs must equal q3_score's bit for bit, and the cache it leaves must
be q3_prefill's."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN_CASES
from qwen3_rs_b200 import transformer as T
from test_gpu_score import bits, check_scores_vs_oracle, kv_rows, lp_bound, lsm64, oracle_logits
from test_gpu_tp import _free_port, _ngpu

pytestmark = pytest.mark.gpu


def topk64(lg, k):
    """float64 reference: ids [rows, k] by (value descending, index descending) and their log-softmax."""
    lg = np.atleast_2d(lg)
    idx = np.arange(lg.shape[1])
    ids = np.stack([np.lexsort((-idx, -r.astype(np.float64)))[:k] for r in lg])
    return ids, np.take_along_axis(lsm64(lg), ids, axis=1)


def check_topk(lg, k, label=""):
    """op_topk_logprobs on lg [rows][n] against topk64 and against op_logprobs (same lp / argmax bits); returns the worst
    relative error of the finite log-probabilities."""
    lg = np.atleast_2d(lg)
    rows, n = lg.shape
    targets = np.random.default_rng(n + k).integers(0, n, rows)
    ids, lps, lp, am = T.op_topk_logprobs(lg, k, targets)
    want_ids, want = topk64(lg, k)
    assert np.array_equal(ids, want_ids), (label, np.argwhere(ids != want_ids)[:5])
    lp1, am1 = T.op_logprobs(lg, targets)
    # k_logprobs' accumulation turns two -inf partials meeting (expf(-inf - -inf)) into s = NaN; the top-k values share m and
    # s with it, so such a row is NaN in both, and only there
    nan = np.isnan(lps).any(axis=1)
    assert np.array_equal(nan, np.isnan(lp1)) and np.isnan(lps[nan]).all(), label
    assert (np.isneginf(lg[nan]).sum(axis=1) >= 2).all(), label
    lps, want = lps[~nan], want[~nan]
    fin = np.isfinite(want)
    assert np.array_equal(np.isneginf(lps), np.isneginf(want)), label
    err = np.abs(lps[fin].astype(np.float64) - want[fin])
    assert (err <= lp_bound(want[fin])).all(), (label, float(err.max()))
    assert np.array_equal(bits(lp), bits(lp1)) and np.array_equal(am, am1), label
    assert np.array_equal(ids[:, 0], am), label
    hit = (ids == targets[:, None])[~nan]  # the target's entry is q3_score's value bit for bit
    assert np.array_equal(bits(lps)[hit], bits(np.broadcast_to(lp[~nan, None], lps.shape))[hit]), label
    return float((err / (1.0 + np.abs(want[fin]))).max()) if err.size else 0.0


# ---- the selection alone --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,n", [(3, 64), (37, 768), (5, 4096), (3, 151936)])
@pytest.mark.parametrize("scale", [1.0, 30.0])
@pytest.mark.parametrize("offset", [0.0, 1e4, -1e4])
def test_op_topk_against_float64(rows, n, scale, offset):
    rng = np.random.default_rng(rows * 7 + n + int(scale) + int(abs(offset)) + (offset < 0))
    lg = (rng.standard_normal((rows, n)) * scale + offset).astype(np.float32)
    worst = max(check_topk(lg, k, f"n {n} k {k}") for k in (1, 20, 64))
    print(f"op_topk rows {rows} n {n} scale {scale} offset {offset}: worst |dlp| / (1 + |lp|) {worst:.2e}")


@pytest.mark.parametrize("k", [1, 7, 64])
def test_op_topk_row_as_wide_as_k(k):
    lg = np.random.default_rng(k).standard_normal((4, k)).astype(np.float32)
    lg[1] = 0.5  # all equal: every index, from the last
    check_topk(lg, k, "n == k")
    ids, _, _, _ = T.op_topk_logprobs(lg[1], k)
    assert ids[0].tolist() == list(range(k - 1, -1, -1))


@pytest.mark.parametrize("n", [256, 5000, 151936])
@pytest.mark.parametrize("k", [1, 20, 64])
def test_op_topk_hard_rows(n, k):
    rng = np.random.default_rng(n * 3 + k)
    rows = []
    rows.append(np.full(n, 0.25, np.float32))                        # all equal: the k largest indices
    r = rng.standard_normal(n).astype(np.float32) - 10.0             # heavy ties straddling the k-th place
    pos = rng.permutation(n)
    r[pos[:k // 2]] = 5.0
    r[pos[k // 2:k // 2 + min(n - k // 2, 3 * k + 50)]] = 2.0
    rows.append(r)
    r = np.full(n, -3.0, np.float32)                                 # top values a few ulps apart: all in one top-digit bin
    m = min(n, 3000)
    r[rng.permutation(n)[:m]] = np.float32(7.0) + (np.arange(m) % 5).astype(np.float32) * np.spacing(np.float32(7.0))
    rows.append(r)
    r = rng.standard_normal(n).astype(np.float32)                    # one -inf: finite log-probabilities
    r[n // 3] = -np.inf
    rows.append(r)
    r = rng.standard_normal(n).astype(np.float32)                    # many -inf entries (log-probabilities NaN, ids exact)
    r[rng.permutation(n)[:n // 2]] = -np.inf
    rows.append(r)
    r = np.full(n, -np.inf, np.float32)                              # fewer finite values than k: -inf among the top k
    r[rng.permutation(n)[:max(1, k // 3)]] = rng.standard_normal(max(1, k // 3)).astype(np.float32)
    rows.append(r)
    r = rng.standard_normal(n).astype(np.float32)                    # one far outlier: the k-th key many bins below the max
    r[n // 2] = 1e30
    rows.append(r)
    lg = np.stack(rows)
    check_topk(lg, k, f"hard rows n {n} k {k}")
    ids, _, _, _ = T.op_topk_logprobs(lg[0], k)
    assert ids[0].tolist() == list(range(n - 1, n - 1 - k, -1))


def test_op_topk_is_deterministic_and_per_row():
    """Reruns give the same bits, and a row launched alone gives the same bits as among 512 rows."""
    rng = np.random.default_rng(17)
    lg = (rng.standard_normal((512, 32768)) * 4).astype(np.float32)
    lg[100] = 1.0
    lg[200, :4000] = 9.0
    tg = rng.integers(0, 32768, 512)
    a = T.op_topk_logprobs(lg, 64, tg)
    b = T.op_topk_logprobs(lg, 64, tg)
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32))
    for r in (0, 100, 200, 511):
        one = T.op_topk_logprobs(lg[r:r + 1], 64, tg[r:r + 1])
        for x, y in zip(one, a):
            assert np.array_equal(np.asarray(x).view(np.uint32)[0], np.asarray(y).view(np.uint32)[r]), r


def test_op_topk_argument_errors_write_nothing():
    lg = np.zeros((2, 256), np.float32)
    ids = np.full((2, 64), -3, np.int32)
    lps = np.full((2, 64), -7.5, np.float32)
    lp = np.full(2, -7.5, np.float32)
    am = np.full(2, -3, np.int32)
    tg = np.array([0, 1], np.int32)
    L = T.load_library()
    p = T._ptr
    for rows, n, k, t, io, vo, lpo in ((2, 256, 0, tg, ids, lps, lp), (2, 256, 65, tg, ids, lps, lp),
                                       (2, 32, 33, tg, ids, lps, lp),                       # k > n
                                       (2, 256, 4, tg, None, lps, lp), (2, 256, 4, tg, ids, None, lp),
                                       (2, 256, 4, None, ids, lps, lp),                     # logprobs without targets
                                       (2, 256, 4, np.array([0, 256], np.int32), ids, lps, lp),
                                       (0, 256, 4, tg, ids, lps, lp), (2, 0, 4, tg, ids, lps, lp)):
        assert L.q3_op_topk_logprobs(0, p(lg), rows, n, k, p(t), p(io), p(vo), p(lpo), p(am)) == -1
        assert (ids == -3).all() and (lps == -7.5).all() and (lp == -7.5).all() and (am == -3).all()


# ---- models -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def topk_models(ckpt):
    cache = {}

    def get(name, gs, seed):
        key = (name, gs, seed)
        if key not in cache:
            cache[key] = T.TransformerBuilder.new(ckpt(name, gs, seed)).build()
        return cache[key]

    yield get
    for m in cache.values():
        m.close()


@pytest.mark.parametrize("name,gs,seed,n,k", [("small", 64, 3, 500, 20), ("wide", 64, 4, 2000, 64)])
def test_score_topk_matches_score(topk_models, name, gs, seed, n, k):
    """Against q3_score on the batched path: the same log-probabilities and argmax bit for bit, ids[:, 0] the argmax, the
    target's top-k entry equal to its log-probability bit for bit, and the cache and next decode step of q3_prefill.  At
    2000 tokens the lm_head runs 4 row chunks, the last one ragged."""
    m = topk_models(name, gs, seed)
    c = m.get_config()
    toks = np.random.default_rng(n + 1).integers(0, c.vocab_size, n + 1).tolist()
    t, tg = toks[:n], toks[1:]
    tg[::7] = [int(x) for x in np.asarray(m.score(t)[1])[::7]]  # every 7th target is the argmax: always in the top k
    m.reset()
    lp, am = m.score(t, targets=tg)
    m.reset()
    ids, lps, lp2, am2 = m.score_topk(t, k, targets=tg)
    kv_topk = kv_rows(m, c.seq_len if c.seq_len <= n + 256 else n + 256)
    nxt_topk = m.forward(toks[n], n)
    assert np.array_equal(bits(lp2), bits(lp)) and np.array_equal(am2, am)
    assert np.array_equal(ids[:, 0], am)
    assert all(len(set(r)) == k for r in ids.tolist()) and (np.diff(lps, axis=1) <= 0).all() and (lps <= 0).all()
    hit = ids == np.asarray(tg)[:, None]
    assert hit[::7].any(axis=1).all()
    assert np.array_equal(bits(lps)[hit], bits(np.broadcast_to(lp[:, None], lps.shape))[hit])
    m.reset()
    ids_b, lps_b, lp_b, am_b = m.score_topk(t, k)  # no targets, and a rerun: the same bits
    assert lp_b is None and np.array_equal(ids_b, ids) and np.array_equal(bits(lps_b), bits(lps)) and np.array_equal(am_b, am)
    m.reset()
    ids_s, lps_s, _, _ = m.score_topk(t, 5, want_argmax=False)  # a smaller k: the first 5 of the same order
    assert np.array_equal(ids_s, ids[:, :5]) and np.array_equal(bits(lps_s), bits(lps[:, :5]))
    m.reset()
    lp3, am3 = m.score(t, targets=tg)  # q3_score after q3_score_topk: unchanged
    assert np.array_equal(bits(lp3), bits(lp)) and np.array_equal(am3, am)
    m.reset()
    m.prefill(t, 0, want_logits=False)
    kv_pf = kv_rows(m, len(kv_topk[0][0]))
    nxt_pf = m.forward(toks[n], n)
    for l, ((kk, v), (kp, vp)) in enumerate(zip(kv_topk, kv_pf)):
        assert np.array_equal(kk, kp) and np.array_equal(v, vp), f"layer {l}: KV rows differ from q3_prefill's"
    assert np.array_equal(bits(nxt_topk), bits(nxt_pf)), "decode after q3_score_topk differs from decode after q3_prefill"


@pytest.mark.parametrize("name,gs,seed", GOLDEN_CASES)
def test_exact_mode_topk_of_the_golden_logits(topk_models, golden, name, gs, seed):
    """Exact mode (sequential forwards, the reference's logits bit for bit): the top k of the golden logits exactly, their
    log-probabilities within the operator bound."""
    key = f"{name}_gs{gs}"
    m = topk_models(name, gs, seed)
    seq = golden[key + "_prompt"].tolist() + golden[key + "_greedy"].tolist()
    lg = golden[key + "_logits"]
    npos, k = lg.shape[0], 20
    m.set_exact(True)
    try:
        m.reset()
        ids, lps, lp, am = m.score_topk(seq[:-1], k, targets=seq[1:])
        m.reset()
        lp1, am1 = m.score(seq[:-1], targets=seq[1:])
    finally:
        m.set_exact(False)
    want_ids, want = topk64(lg, k)
    assert np.array_equal(ids[:npos], want_ids)
    assert (np.abs(lps[:npos].astype(np.float64) - want) <= lp_bound(want)).all()
    assert np.array_equal(bits(lp), bits(lp1)) and np.array_equal(am, am1) and np.array_equal(ids[:, 0], am)


@pytest.mark.parametrize("name,gs,seed,n", [("tiny-untied", 64, 1, 37), ("small", 128, 2, 130)])
def test_fast_path_topk_matches_oracle(topk_models, ckpt, name, gs, seed, n):
    """The batched path against the oracle's sequential forwards.  Every returned log-probability is within the bound
    test_gpu_score sets for q3_score of the oracle's value for that id, and within twice that of the oracle's value at the same
    rank; where the oracle's gaps to both neighbouring ranks exceed twice the bound, the id is the oracle's."""
    m = topk_models(name, gs, seed)
    k = 20
    toks = np.random.default_rng(n + 11).integers(0, m.get_config().vocab_size, n + 1).tolist()
    path = ckpt(name, gs, seed)
    lo, lo2 = oracle_logits(path, toks[:n], 0), oracle_logits(path, toks[:n], 1)
    m.reset()
    ids, lps, lp, am = m.score_topk(toks[:n], k, targets=toks[1:])
    check_scores_vs_oracle(lp, am, lo, lo2, np.array(toks[1:]), f"{name} gs{gs} T {n} (top-k call)")
    bound = 2 * (0.05 * float(np.abs(lo).max()) + 1e-2)
    lsm = lsm64(lo)
    got = np.take_along_axis(lsm, ids.astype(np.int64), axis=1)
    assert (np.abs(lps - got) <= bound).all()
    o_ids, o_lps = topk64(lo, k + 1)
    assert (np.abs(got - o_lps[:, :k]) <= 2 * bound).all()
    gap_hi = np.concatenate([np.full((n, 1), np.inf), o_lps[:, :k - 1] - o_lps[:, 1:k]], axis=1)
    gap_lo = o_lps[:, :k] - o_lps[:, 1:k + 1]
    sure = (gap_hi > 2 * bound) & (gap_lo > 2 * bound)
    assert np.array_equal(ids[sure], o_ids[:, :k][sure])
    print(f"{name} gs{gs} T {n}: {int(sure.sum())} of {n * k} ranks clear of the noise, all equal to the oracle's")


def test_score_topk_argument_errors_write_nothing(topk_models):
    m = topk_models("small", 64, 3)
    c = m.get_config()
    L = T.load_library()
    p = T._ptr
    toks = np.arange(1, 9, dtype=np.int32)
    tg = np.arange(2, 10, dtype=np.int32)
    ids = np.full((8, 64), -3, np.int32)
    lps = np.full((8, 64), -7.5, np.float32)
    lp = np.full(8, -7.5, np.float32)
    am = np.full(8, -3, np.int32)
    bad_tok = toks.copy()
    bad_tok[5] = c.vocab_size
    bad_tg = tg.copy()
    bad_tg[7] = -1
    h = C.c_void_p(m._h)
    cases = [(toks, 8, 0, 0, ids, lps, tg, lp), (toks, 8, 0, 65, ids, lps, tg, lp), (toks, 8, 0, -1, ids, lps, tg, lp),
             (toks, 8, 0, 4, None, lps, tg, lp), (toks, 8, 0, 4, ids, None, tg, lp), (toks, 8, 0, 4, ids, lps, None, lp),
             (toks, 8, 0, 4, ids, lps, bad_tg, lp), (bad_tok, 8, 0, 4, ids, lps, tg, lp), (toks, 0, 0, 4, ids, lps, tg, lp),
             (toks, 8, c.seq_len - 7, 4, ids, lps, tg, lp), (toks, 8, -1, 4, ids, lps, tg, lp)]
    for tk, n, pos0, k, io, vo, tgt, lpo in cases:
        assert L.q3_score_topk(h, p(tk), n, pos0, k, p(io), p(vo), p(tgt), p(lpo), p(am)) == -1, (n, pos0, k)
        assert (ids == -3).all() and (lps == -7.5).all() and (lp == -7.5).all() and (am == -3).all()
    m.reset()
    ids_ok, _, lp_ok, _ = m.score_topk(toks.tolist(), 64, targets=tg.tolist())  # the handle stays usable
    assert np.isfinite(lp_ok).all() and (ids_ok >= 0).all()


# ---- tensor parallel ----------------------------------------------------------------------------------------------------
def _tp_worker(rank, world, port, path, n, k, q):
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        m = T.TransformerBuilder.new(path).with_device(rank).with_tensor_parallel(rank, world).build()
        T.tp_connect(m, dist)
        toks = np.random.default_rng(n).integers(0, m.get_config().vocab_size, n + 1).tolist()
        ids, lps, lp, am = m.score_topk(toks[:n], k, targets=toks[1:])
        code = 0
        try:
            m.set_exact(True)
            m.score_topk(toks[:n], k)
        except T.Q3Error as e:
            code = e.code
        q.put((rank, {"ids": ids, "lps": lps, "lp": lp, "am": am, "toks": toks, "exact_code": code}))
        dist.barrier()
        m.close()
    except Exception as e:  # noqa: BLE001 -- surface the failure to the parent instead of a queue timeout
        import traceback

        q.put((rank, {"error": repr(e) + "\n" + traceback.format_exc()}))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("name,gs,seed,world", [("small", 64, 3, 2), ("small8", 64, 5, 4)])
def test_tensor_parallel_topk(ckpt, name, gs, seed, world):
    """Every rank runs the full lm_head: the ranks' results are bit-identical, and the ids are one GPU's wherever one GPU's
    log-probabilities clear both neighbouring ranks by 0.5 (the partial blocks are summed in another order than on one GPU, as
    test_gpu_score allows for the argmax).  Exact mode under tensor parallelism: Q3_EUNSUPPORTED."""
    import torch.multiprocessing as mp

    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    path, n, k = ckpt(name, gs, seed), 120, 20
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_tp_worker, args=(r, world, port, path, n, k, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    got = dict(q.get(timeout=240) for _ in range(world))
    for pr in procs:
        pr.join(60)
    for r in range(world):
        assert "error" not in got[r], got[r]["error"]
        assert got[r]["exact_code"] == -5
    for r in range(1, world):
        for f in ("ids", "lps", "lp", "am"):
            assert np.array_equal(np.asarray(got[r][f]).view(np.uint32), np.asarray(got[0][f]).view(np.uint32)), (r, f)
    toks = got[0]["toks"]
    m = T.TransformerBuilder.new(path).build()
    try:
        ids1, lps1, _, _ = m.score_topk(toks[:n], k + 1)
    finally:
        m.close()
    assert np.array_equal(got[0]["ids"][:, 0], got[0]["am"])
    gap_hi = np.concatenate([np.full((n, 1), np.inf), lps1[:, :k - 1] - lps1[:, 1:k]], axis=1)
    gap_lo = lps1[:, :k] - lps1[:, 1:k + 1]
    sure = (gap_hi > 0.5) & (gap_lo > 0.5)
    print(f"{name} tp{world}: {(ids1[:, :k] == got[0]['ids']).mean():.4f} of the ids equal one GPU's; {int(sure.sum())} clear ranks")
    assert np.array_equal(got[0]["ids"][sure], ids1[:, :k][sure])
