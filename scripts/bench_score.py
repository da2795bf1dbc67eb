"""q3_score at T 2048 on synthetic Qwen3-4B / 8B gs64 checkpoints (quantised on the device, as bench.py does).

Per model, one JSON line:
  prefill_ms        q3_bench_prefill (CUDA events, the batched forward without the head), median of --reps
  score_ms          host clock around the synchronous q3_score call (log-probabilities + argmax of all T positions), median
                    of --reps after one warm-up call
  head_ms           score_ms - prefill_ms: final norm + lm_head GEMM + reduction on every row, plus the call's copies
  head_int8_TOPS    2 T vocab dim / head_ms
  lm_head_gemm_ms   the lm_head GEMM alone in the same row chunks (q3_bench_gemm_q8, best of reps), for the split of head_ms
  scored_tok_s      T / score_ms
  forward_ms_per_token  256 sequential q3_forward calls with host logits (the way to get the same numbers without q3_score)
With --topk K1,K2,..: q3_score_topk with targets at each k, timed like score_ms with the calls of every k and q3_score's
alternated rep by rep (topk_ms, median; topk_extra_ms = topk_ms - the alternated q3_score's median).
The card's name, power limit and max SM clock are read in the same run.

usage: python scripts/bench_score.py [--models qwen3-4b,qwen3-8b] [--T 2048] [--reps 7] [--topk 1,20,64]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from qwen3_rs_b200 import synth, transformer as T  # noqa: E402

SCORE_ROWS = 512  # q3_engine.cu: lm_head rows per GEMM


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        import torch

        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e!r})"}


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def run_topk(m, t, tg, ks, reps):
    """q3_score and q3_score_topk at every k, alternated rep by rep after one warm-up call each."""
    fns = {0: lambda: m.score(t, targets=tg)}
    for k in ks:
        fns[k] = lambda k=k: m.score_topk(t, k, targets=tg)
    for f in fns.values():
        f()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            ms[k].append(timed(f)[0])
    base = float(np.median(ms[0]))
    return {"topk_score_ms": base, "topk_ms": {k: float(np.median(ms[k])) for k in ks},
            "topk_extra_ms": {k: float(np.median(ms[k])) - base for k in ks}, "topk_ms_all": {k: ms[k] for k in ks}}


def run(model, Tn, reps, ks=()):
    shape = synth.SHAPES[model]
    m = T.TransformerBuilder.new(bench.bench_checkpoint(model, 64)).with_ctx_length(Tn + 8).build()
    try:
        toks = np.random.default_rng(0).integers(0, shape.vocab_size, Tn + 1).tolist()
        t, tg = toks[:Tn], toks[1:]
        pf = [m.bench_prefill(t, 0) for _ in range(reps)]
        m.score(t, targets=tg)  # warm-up: sizes the lm_head buffers
        sc = []
        for _ in range(reps):
            t0 = time.perf_counter()
            lp, am = m.score(t, targets=tg)
            sc.append((time.perf_counter() - t0) * 1e3)
        pf_ms, sc_ms = float(np.median(pf)), float(np.median(sc))
        head_ms = sc_ms - pf_ms
        ops = 2.0 * Tn * shape.vocab_size * shape.dim
        gemm_ms = 0.0
        for r0 in range(0, Tn, SCORE_ROWS):
            gemm_ms += T.bench_gemm_q8(min(SCORE_ROWS, Tn - r0), shape.vocab_size, shape.dim, 64, 0, reps)
        topk = run_topk(m, t, tg, ks, reps) if ks else {}
        m.reset()
        lg = np.empty(shape.vocab_size, np.float32)
        m.forward(t[0], 0)
        t0 = time.perf_counter()
        for p in range(256):
            lg = m.forward(t[p], p)
        fwd_ms = (time.perf_counter() - t0) * 1e3 / 256
        return {"model": model, "group_size": 64, "T": Tn, "prefill_ms": pf_ms, "score_ms": sc_ms, "score_ms_all": sc,
                "head_ms": head_ms, "head_int8_TOPS": ops / head_ms / 1e9, "lm_head_gemm_ms": gemm_ms,
                "lm_head_gemm_int8_TOPS": ops / gemm_ms / 1e9, "scored_tok_s": Tn / sc_ms * 1e3,
                "forward_ms_per_token": fwd_ms, "mean_logprob": float(np.mean(lp)), "finite": bool(np.isfinite(lp).all() and np.isfinite(lg).all()), **topk}
    finally:
        m.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", default="qwen3-4b,qwen3-8b")
    ap.add_argument("--T", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--topk", default="", help="comma-separated k values for q3_score_topk, e.g. 1,20,64")
    a = ap.parse_args()
    ks = [int(k) for k in a.topk.split(",") if k]
    info = card()
    for model in a.models.split(","):
        bench.emit({**run(model, a.T, a.reps, ks), **info})


if __name__ == "__main__":
    main()
