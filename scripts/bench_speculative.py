"""q3_forward_multi and q3_decode_speculative on a synthetic Qwen3-8B gs64 target (quantised on the device, as bench.py does).

JSON lines:
  step      per position: q3_bench_multi for n = 1, 2, 4, 8 (ms per call, and relative to one graph step), the single-token graph
            step and the persistent step (q3_bench_decode over --steps consecutive positions), CUDA events
  spec      per draft and k: decode_speculative tokens/s over --n tokens after a --prompt token prefill (host clock around the
            synchronous call, so the per-round host work is included), its rounds / drafted / accepted, and decode_greedy's
            tokens/s on the graph and persistent paths from the same cache state
  projection  tokens/s as a function of the acceptance rate a, from the measured costs: a round of k drafted tokens costs
            k * draft_step + verify(k + 1) + host overhead (measured with the 0.6B draft) and emits (1 - a^(k+1)) / (1 - a)
            tokens on average (independent acceptances).  A projection: random-init weights cannot show real acceptance rates.
Drafts: the synthetic Qwen3-0.6B on the persistent path (acceptance near 0: the overhead floor) and a second handle on the 8B
checkpoint on the multi-kernel path, whose tokens are the verifier's bit for bit (acceptance 1).
The card's name, power limit and max SM clock are read in the same run.

usage: python scripts/bench_speculative.py [--positions 512,4096] [--reps 50] [--steps 64] [--n 256] [--prompt 512] [--ks 1,3,7]"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from qwen3_rs_b200 import transformer as T  # noqa: E402
from scripts.bench_score import card  # noqa: E402


def step_costs(m, pos, reps, steps):
    out = {"pos": pos}
    for n in (1, 2, 4, 8):
        out[f"multi_{n}_ms"] = m.bench_multi(n, pos, reps) / reps
    m.set_decode_path(0)
    out["graph_step_ms"] = m.bench_decode(0, pos, steps) / steps
    m.set_decode_path(1)
    out["persistent_step_ms"] = m.bench_decode(0, pos, steps) / steps
    for n in (1, 2, 4, 8):
        out[f"multi_{n}_over_graph"] = out[f"multi_{n}_ms"] / out["graph_step_ms"]
    return out


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--positions", default="512,4096")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--prompt", type=int, default=512)
    ap.add_argument("--ks", default="1,3,7")
    a = ap.parse_args()
    info = card()
    positions = [int(p) for p in a.positions.split(",")]
    ks = [int(k) for k in a.ks.split(",")]
    ctx = max(max(positions) + a.steps + 16, a.prompt + a.n + 16)
    path8, path06 = bench.bench_checkpoint("qwen3-8b", 64), bench.bench_checkpoint("qwen3-0.6b", 64)
    tgt = T.TransformerBuilder.new(path8).with_ctx_length(ctx).build()
    twin = T.TransformerBuilder.new(path8).with_ctx_length(ctx).build()
    small = T.TransformerBuilder.new(path06).with_ctx_length(ctx).build()
    try:
        steps = {}
        for p in positions:
            steps[p] = step_costs(tgt, p, a.reps, a.steps)
            bench.emit({"kind": "step", "model": "qwen3-8b", "group_size": 64, **steps[p], **info})
        small.set_decode_path(0)
        small_graph = small.bench_decode(0, a.prompt, a.steps) / a.steps
        small.set_decode_path(1)
        small_persistent = small.bench_decode(0, a.prompt, a.steps) / a.steps
        prompt = np.random.default_rng(0).integers(0, 151936, a.prompt).tolist()
        for m in (tgt, twin, small):
            m.reset()
            m.prefill(prompt[:-1], 0, want_logits=False)
        first, pos0 = prompt[-1], a.prompt - 1
        base = {}
        for path in (0, 1):
            tgt.set_decode_path(path)
            tgt.decode_greedy(first, pos0, 8)  # warm-up
            ms, want = timed(lambda: tgt.decode_greedy(first, pos0, a.n))
            base[path] = a.n / ms * 1e3
        tgt.set_decode_path(1)
        overhead = {}
        for name, draft, path in (("qwen3-0.6b", small, 1), ("qwen3-8b twin", twin, 0)):
            draft.set_decode_path(path)
            for k in ks:
                tgt.decode_speculative(draft, first, pos0, 2 * (k + 1), k)  # warm-up: captures the graphs
                ms, (got, st) = timed(lambda: tgt.decode_speculative(draft, first, pos0, a.n, k))
                rate = a.n / ms * 1e3
                row = {"kind": "spec", "target": "qwen3-8b", "draft": name, "k": k, "n": a.n, "pos0": pos0, "tok_s": rate, "ms": ms,
                       **st, "acceptance": st["accepted"] / max(st["drafted"], 1), "greedy_graph_tok_s": base[0],
                       "greedy_persistent_tok_s": base[1], **info}
                if name == "qwen3-0.6b":
                    draft_ms = small_persistent
                    verify_ms = tgt.bench_multi(k + 1, pos0, a.reps) / a.reps
                    overhead[k] = (ms - st["drafted"] * draft_ms - st["rounds"] * verify_ms) / st["rounds"]
                    row.update({"draft_step_ms": draft_ms, "verify_ms": verify_ms, "host_overhead_ms_per_round": overhead[k]})
                bench.emit(row)
        tgt.set_decode_path(0)
        ref = tgt.decode_greedy(first, pos0, a.n)
        got, _ = tgt.decode_speculative(small, first, pos0, a.n, ks[-1])
        bench.emit({"kind": "check", "speculative_equals_graph_greedy": got == ref, "n": a.n})
        for k in ks:
            verify = tgt.bench_multi(k + 1, pos0, a.reps) / a.reps
            rows = {}
            for acc in (0.0, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0):
                tokens = k + 1 if acc == 1.0 else (1 - acc ** (k + 1)) / (1 - acc)
                # the extra draft step of a fully accepted round is one more draft step
                cost = k * small_persistent + verify + overhead.get(k, 0.0) + (acc ** k) * small_persistent
                rows[str(acc)] = tokens / cost * 1e3
            bench.emit({"kind": "projection", "k": k, "draft": "qwen3-0.6b (persistent path)", "draft_step_ms": small_persistent,
                        "draft_graph_step_ms": small_graph, "verify_ms": verify, "host_overhead_ms_per_round": overhead.get(k),
                        "tok_s_by_acceptance": rows, "greedy_persistent_tok_s": base[1], **info})
    finally:
        for m in (tgt, twin, small):
            m.close()


if __name__ == "__main__":
    main()
