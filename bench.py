#!/usr/bin/env python
"""bench.py -- Qwen3 Q8 batch-1 decode throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    python bench.py --gpus 1 ... --dump-outputs DIR           # also write the last timed step's tokens / logits as .npy

One "step" = `--tokens-per-step` (default 64) greedy decode tokens of the named model, batch 1.
Workload at N=1: Qwen3-8B architecture, random-init weights exported with group size 64 through
the repo's exporter (no checkpoints offline), i.e. BASELINE.json configs[3] at one GPU.

  value   : decode tokens/s, whole job, device-timed (CUDA events on the launch stream inside
            q3_bench_decode, cross-checked by a host clock around barrier+synchronize), token
            feedback on the device, weights/KV resident in HBM.
  e2e     : the same tokens/s through the reference-facing call -- Transformer.forward(token, pos)
            -> host logits (vocab x f32 D2H every token) -> host argmax (sampler.rs semantics),
            over the SAME positions as `value` (the cache below them is refilled untimed).
  parity  : (N=1) the GPU against the CPU oracle on the bench checkpoint itself, teacher-forced along
            the oracle's greedy tokens: max |dlogit| and token agreement in exact (reference-order) mode
            and in the fast mode that `value` times, plus exact mode's own tokens/s.
  long_context / prefill_4b: BASELINE.json configs 5 and 3 (32K-token KV cache decode; Qwen3-4B
            2048-token batched prefill + 256 decode tokens), N=1 only, skipped with --no-extras.
  roofline: the dominant kernel.  On the default path the whole decode step is ONE launch of the
            persistent kernel k_mega_decode, so algorithmic bytes per launch = bytes per token
            (weights + scales + f32 KV rows read) and the duration is the CUDA-event time per launch
            over the timed region; peak = MEASURED_PEAKS.json's HBM copy bandwidth.  `graph_path_kernels`
            lists the multi-kernel path's GEMVs timed alone for comparison.
  cpu_baseline: the CPU oracle (C restatement of the reference forward, OpenMP over rows/heads
            like the reference's rayon) on the same .bin and the box's host cores, bounded sample.

Prints exactly one JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Exactly ONE JSON line may reach stdout, but native libraries write there too (NCCL prints its version
# banner to fd 1).  So fd 1 is pointed at stderr for the whole run and the result line goes to a saved
# duplicate of the original stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj) -> None:
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


# ---------------------------------------------------------------------------------------------
# checkpoint (synthetic, exported by the repo's exporter)
# ---------------------------------------------------------------------------------------------
def bench_checkpoint(model: str, gs: int, seed: int = 0) -> str:
    from qwen3_rs_b200 import synth

    shape = synth.SHAPES[model]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    d = os.path.join(base, f"q3_bench-{os.getuid()}")  # per user: another user's cache directory is not writable
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"{model}_gs{gs}_s{seed}.bin")
    want = synth.checkpoint_bytes(shape, gs)
    if os.path.exists(path) and os.path.getsize(path) == want:
        return path
    t0 = time.time()
    try:
        import torch

        cuda = torch.cuda.is_available()
    except Exception:
        cuda = False
    tmp = path + f".tmp{os.getpid()}"
    if cuda:
        # weights generated on the GPU and quantised by the library's own exporter kernel (k_quantize_q80, SURVEY 8f-3;
        # bit-identical to export.quantize_q80: tests/test_gpu_parity.py::test_device_quantizer_makes_identical_checkpoints)
        synth.export_synthetic(shape, tmp, gs, seed=seed, device="cuda", quantizer=synth.quantize_q80_device)
    else:
        synth.export_synthetic(shape, tmp, gs, seed=seed)
    os.replace(tmp, path)
    log(f"[bench] exported {model} gs{gs} -> {path} ({want / 1e9:.2f} GB) in {time.time() - t0:.1f}s")
    return path


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                smax.append(float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kind: str, workload: str = ""):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture; null when the capture
    was taken on another workload (model / group size / GPUs) than the one being timed."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            d = json.load(f)
        return d.get(kind) if d.get("workload", "") == workload else None
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline (the oracle; the only place bench.py executes oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_decode_tok_s(path: str, ctx: int, n_tokens: int, threads: int = 0):
    """-> tok/s, threads, seconds, input tokens [n+1], logits [n+1][vocab] of the oracle's greedy run from token 1."""
    from oracle import binding as orc

    orc.set_threads(threads or os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1: use every host core
    cores = orc.max_threads()
    m = orc.Model(path, ctx)
    tok = 1
    seq, logits = [tok], []
    lg = m.forward(tok, 0)  # untimed first touch (page-in of the mmap)
    logits.append(lg)
    tok = orc.argmax(lg)
    t0 = time.perf_counter()
    for pos in range(1, 1 + n_tokens):
        seq.append(tok)
        lg = m.forward(tok, pos)
        logits.append(lg)
        tok = orc.argmax(lg)
    dt = time.perf_counter() - t0
    m.close()
    return n_tokens / dt, cores, dt, seq, np.stack(logits)


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    path = bench_checkpoint(args.model, args.group_size)
    # bounded sample: a few tokens per step so the whole run stays within minutes
    tps = max(1, min(args.tokens_per_step, args.ref_tokens_per_step))
    from oracle import binding as orc

    orc.set_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1: use every host core
    cores = orc.max_threads()
    m = orc.Model(path, args.ctx)
    # Same positions as the CUDA arm's timed region: step i starts at (warmup + i) * tokens_per_step; of each step's
    # tokens_per_step tokens the first `tps` are run (the CPU decodes ~5 tok/s: a full 64-token step takes ~13 s).  The
    # cache below the sampled positions holds whatever the sampled tokens wrote, zeros elsewhere -- the arithmetic per
    # token (all weights once + attention over pos+1 rows) does not depend on the values.
    tok = 1
    for w in range(args.warmup):
        tok = orc.argmax(m.forward(tok, w * args.tokens_per_step))
    t0 = time.perf_counter()
    for i in range(args.steps):
        pos = (args.warmup + i) * args.tokens_per_step
        for _ in range(tps):
            tok = orc.argmax(m.forward(tok, pos))
            pos += 1
    dt = time.perf_counter() - t0
    val = args.steps * tps / dt
    sample = (f"{args.steps} steps x the first {tps} of each step's {args.tokens_per_step} greedy tokens of {args.model} gs{args.group_size}, at the CUDA "
              f"arm's positions ({args.warmup * args.tokens_per_step}..); {cores} OpenMP threads")
    out = {
        "impl": "reference", "metric": "decode_tokens_per_s", "value": val, "unit": "tok/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        # time of one full tokens_per_step-token step at the measured rate (tokens_run_per_step were actually run and timed)
        "ms_per_step": dt / args.steps * 1e3 * (args.tokens_per_step / tps), "tokens_run_per_step": tps,
        "ms_per_sampled_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int8 weights x int8 activations, int32 group dots, f32 accumulate",
        "data": "synthetic", "config": workload_config(args), "parallelism": "host threads", "where": "cpu",
        "cpu_baseline": {"value": val, "unit": "tok/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = C restatement of qwen3-rs's CPU forward (oracle/q3_oracle.c); the Rust toolchain is absent so the reference itself cannot be built",
    }
    emit(out)


def workload_config(args) -> dict:
    """The workload only -- identical for both arms and every N (how it is run goes into top-level keys)."""
    return {
        "workload": f"{args.model} Q8_0 group_size {args.group_size}, batch-1 greedy decode, {args.tokens_per_step} tokens/step, ctx {args.ctx}",
        "checkpoint": args.model, "group_size": args.group_size, "ctx": args.ctx, "tokens_per_step": args.tokens_per_step,
        "l2": "weights streamed per token (>= 0.6 GB) exceed the 126 MB L2; no explicit flush",
        "weights": "random-init, seeded, exported by qwen3_rs_b200.export (reference .bin format)",
    }


# ---------------------------------------------------------------------------------------------
# parity on the bench checkpoint; BASELINE.json configs 5 and 3 (N=1 extras)
# ---------------------------------------------------------------------------------------------
def parity_block(m, oseq, ologits, args) -> dict:
    """GPU vs the CPU oracle on the timed checkpoint, teacher-forced along the oracle's greedy tokens (so nothing but the
    forward arithmetic is compared): exact mode (reference-order reductions; expected bit-identical) and the fast mode
    that `value` times.  north_star: logits max-abs <= 1e-2, greedy tokens identical."""
    from qwen3_rs_b200.sampler import argmax_last

    n = len(oseq)
    want = [int(np.argmax(ologits[p])) for p in range(n)]
    out = {"checkpoint": f"{args.model} gs{args.group_size}", "positions": n, "reference": "oracle/q3_oracle.c (C restatement of the reference forward)",
           "tolerance": {"logits_max_abs": 1e-2, "tokens": "identical"}}
    for mode in ("exact", "fast"):
        m.set_exact(mode == "exact")
        m.reset()
        errs, same = [], 0
        t0 = time.perf_counter()
        outs = [m.forward(oseq[p], p) for p in range(n)]
        dt = time.perf_counter() - t0
        for p in range(n):
            errs.append(float(np.abs(outs[p] - ologits[p]).max()))
            same += int(argmax_last(outs[p]) == argmax_last(ologits[p]))
        out[mode] = {"max_abs_dlogit": max(errs), "max_abs_dlogit_per_position": errs, "tokens_identical": same == n, "tokens_agree": f"{same}/{n}",
                     "tok_s": n / dt, "within_tolerance": max(errs) <= 1e-2 and same == n}
    m.set_exact(False)
    out["logit_scale"] = float(np.abs(ologits).max())
    out["note"] = ("fast mode = identical int32 group dots and per-group terms, parallel f32 reduction trees; a last-ulp difference can flip one int8 "
                   "activation, which later layers amplify on random-init weights (DESIGN.md section 2) -- exact mode is the bit-level proof")
    return out


def long_context_line(path, args, shape, peak, device) -> dict:
    """BASELINE.json config 5: batch-1 decode against a 32 768-token f32 KV cache (split-K GQA attention)."""
    from qwen3_rs_b200 import transformer as T

    npos, steps = 32768, 24
    m = T.TransformerBuilder.new(path).with_ctx_length(npos + steps + 8).with_device(device).build()
    try:
        c = m.get_config()
        kvd = c.n_kv_heads * c.head_dim
        rng = np.random.default_rng(5)
        blk = rng.standard_normal((4096, kvd)).astype(np.float32)
        for l in range(c.n_layers):  # synthetic N(0,1) K / V rows (SURVEY 8d), tiled
            for p0 in range(0, npos, 4096):
                m.kv_write(l, p0, blk, blk)
        m.bench_decode(1, npos, 4)
        ms = min(m.bench_decode(1, npos + 4, steps - 4) for _ in range(2)) / (steps - 4)
        btok = shape.bytes_per_token(args.group_size, npos + steps // 2)
        return {"workload": f"{args.model} gs{args.group_size} decode at positions {npos + 4}..{npos + steps} (32K-token f32 KV cache, synthetic N(0,1) rows)",
                "value": 1e3 / ms, "unit": "tok/s", "us_per_token": ms * 1e3, "bytes_per_token": btok, "achieved_GBps": btok / ms / 1e6,
                "frac_of_measured_peak": btok / ms / 1e6 / peak, "frac_of_8TBps": btok / ms / 1e6 / 8000.0}
    finally:
        m.close()


def prefill_4b_line(args, device) -> dict:
    """BASELINE.json config 3: Qwen3-4B gs64, 2048-token batched prefill (tcgen05 int8 GEMM) + 256 decode tokens."""
    from qwen3_rs_b200 import synth, transformer as T

    shape = synth.SHAPES["qwen3-4b"]
    path = bench_checkpoint("qwen3-4b", 64)
    m = T.TransformerBuilder.new(path).with_ctx_length(2048 + 256 + 8).with_device(device).build()
    try:
        Tn = 2048
        toks = np.random.default_rng(0).integers(0, shape.vocab_size, Tn).tolist()
        pms = m.bench_prefill(toks, 0)
        ah, kvd = shape.n_heads * shape.head_dim, shape.n_kv_heads * shape.head_dim
        ops = 2.0 * Tn * shape.n_layers * (2 * shape.dim * ah + 2 * shape.dim * kvd + 3 * shape.dim * shape.hidden_dim)
        m.bench_decode(1, Tn, 8)
        dms = m.bench_decode(1, Tn, 256) / 256
        btok = shape.bytes_per_token(64, Tn + 128)
        return {"workload": "qwen3-4b gs64: 2048-token prefill + 256 decode tokens", "prefill_tok_s": Tn / pms * 1e3, "prefill_ms": pms,
                "gemm_int8_TOPS": ops / pms / 1e9, "frac_of_int8_peak_4500_TOPS_spec": ops / pms / 1e9 / 4500.0,
                "decode_tok_s": 1e3 / dms, "decode_frac_of_8TBps": btok / dms / 1e6 / 8000.0}
    finally:
        m.close()


# ---------------------------------------------------------------------------------------------
# outputs of the timed path (--dump-outputs)
# ---------------------------------------------------------------------------------------------
def device_logits(m) -> np.ndarray:
    """The handle's device logits buffer (q3_logits_device) copied to the host without running a step: the logits the
    last decode step computed."""
    import types

    import torch

    from qwen3_rs_b200 import transformer as T

    ptr = T.load_library().q3_logits_device(m._h)
    buf = types.SimpleNamespace(__cuda_array_interface__={
        "shape": (m.get_config().vocab_size,), "typestr": "<f4", "data": (ptr, False), "version": 2})
    return torch.as_tensor(buf, device="cuda").cpu().numpy()


def dump_last_step(m, tok0: int, pos0: int, tps: int, out_dir: str) -> None:
    """Writes what the last timed step (q3_bench_decode: tps greedy tokens from tok0 at pos0) computed: decode_logits.npy,
    the logits of its last position read from the device, and decode_tokens.npy, its greedy tokens.  q3_bench_decode keeps
    the tokens on the device, so the step is run once more through q3_decode_greedy (the same launches on the same cache);
    the rerun must leave bit-identical logits, or the tokens would not be the timed step's."""
    logits = device_logits(m)
    tokens = np.array(m.decode_greedy(tok0, pos0, tps), np.float64)
    if not np.array_equal(device_logits(m), logits):
        raise SystemExit("bench.py: the last timed step, run again, computed other logits")
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "decode_logits.npy"), logits)
    np.save(os.path.join(out_dir, "decode_tokens.npy"), tokens)


# ---------------------------------------------------------------------------------------------
# main arm
# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="qwen3-8b")
    ap.add_argument("--group-size", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=2048)
    ap.add_argument("--tokens-per-step", type=int, default=64)
    ap.add_argument("--ref-tokens-per-step", type=int, default=4)
    ap.add_argument("--no-extras", action="store_true", help="skip the parity block, the 32K-context line and the 4B prefill line")
    ap.add_argument("--cpu-sample-tokens", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefill", action="store_true")
    ap.add_argument("--decode-path", type=int, default=-1)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's greedy tokens and last logits as DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        raise SystemExit("bench.py: --dump-outputs writes the CUDA path's outputs on one GPU (--impl ours, no torchrun)")
    need = (args.steps + args.warmup) * args.tokens_per_step + 8
    if args.ctx < need:
        args.ctx = need

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from qwen3_rs_b200 import synth, transformer as T
    from qwen3_rs_b200.sampler import argmax_last

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the forward path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shape = synth.SHAPES[args.model]
    if rank == 0:
        path = bench_checkpoint(args.model, args.group_size)
    barrier()
    path = bench_checkpoint(args.model, args.group_size)

    b = T.TransformerBuilder.new(path).with_ctx_length(args.ctx).with_device(local_rank)
    tp = world
    if tp > 1:
        b = b.with_tensor_parallel(rank, tp)
    m = b.build()
    if tp > 1:
        T.tp_connect(m, dist)
    if args.decode_path >= 0:
        m.set_decode_path(args.decode_path)
    tps = args.tokens_per_step

    # ---- device-timed: value ----
    tok0 = 1
    pos = 0
    for _ in range(args.warmup):
        m.bench_decode(tok0, pos, tps)
        pos += tps
    clocks = ClockSampler(local_rank)
    barrier()
    clocks.start()
    t0 = time.perf_counter()
    dev_ms = 0.0
    pos_start = pos
    for _ in range(args.steps):
        dev_ms += m.bench_decode(tok0, pos, tps)
        pos += tps
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clk = clocks.stop()
    times = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = times.tolist()
    n_tok = args.steps * tps
    value = n_tok / (dev_ms / 1e3)
    if args.dump_outputs:
        dump_last_step(m, tok0, pos - tps, tps, args.dump_outputs)

    # ---- end to end through the reference-facing call: forward -> host logits -> host argmax ----
    # same positions as `value`: the cache below pos_start is refilled untimed, then every one of the n_tok
    # positions is decoded through Transformer.forward
    m.reset()
    for p0 in range(0, pos_start, tps):
        m.bench_decode(tok0, p0, min(tps, pos_start - p0))
    tok, p = tok0, pos_start
    e2e_tokens = n_tok
    if world > 1:
        # the caller lives on rank 0: it alone receives the full-vocabulary logits (the other ranks push their shard to it and
        # take the same token from the device argmax -- identical by construction, checked below)
        m.tp_set_logits_root(0)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_tokens):
        tok = argmax_last(m.forward(tok, p, copy=False)) if rank == 0 else m.forward_argmax(tok, p)  # a borrow, as the reference returns
        p += 1
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = e2e_tokens / e2e_t.item()
    if world > 1:
        m.tp_set_logits_root(-1)
        toks = torch.tensor([tok], dtype=torch.int64, device="cuda")
        lo, hi = toks.clone(), toks.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        if lo.item() != hi.item():
            raise SystemExit("bench.py: tensor-parallel ranks diverged in the end-to-end loop")

    # ---- batched prefill, timed here because every rank of a tensor-parallel group takes part (partial blocks reduced over NVLink) ----
    pms, prefill_err = None, None
    if not args.no_prefill:
        try:
            Tn = min(2048, args.ctx)
            ptoks = np.random.default_rng(0).integers(0, shape.vocab_size, Tn).tolist()
            m.reset()
            pms = m.bench_prefill(ptoks, 0)
        except Exception as e:  # noqa: BLE001
            prefill_err = str(e)
            pms = float("nan")
        if world > 1:
            tms = torch.tensor([pms], device="cuda")
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            pms = float(tms.item())

    if rank != 0:
        m.close()
        if world > 1:
            dist.destroy_process_group()
        return

    vocab = m.get_config().vocab_size
    # ---- roofline ----
    peak, peak_src = measured_peak_gbs()
    mean_pos = pos_start + (n_tok - 1) / 2.0
    btok = shape.bytes_per_token(args.group_size, int(mean_pos)) / tp
    tok_ms = dev_ms / n_tok
    token_roof = {"bytes_per_token_per_gpu": btok, "achieved": btok / tok_ms / 1e6, "peak": peak, "unit": "GB/s",
                  "frac": btok / tok_ms / 1e6 / peak, "frac_of_8TBps": btok / tok_ms / 1e6 / 8000.0,
                  "us_per_token": tok_ms * 1e3, "mean_pos": mean_pos}
    roof = None
    kernels = {}
    launches_per_token = m.launches_per_step  # on the path that was timed (1 for the persistent kernel)
    persistent = launches_per_token == 1
    try:
        if persistent:
            # the whole decode step is ONE launch of k_mega_decode: algorithmic bytes per launch = bytes per
            # token (weights + scales + f32 KV rows read), duration = CUDA-event time per launch measured
            # over the timed region above
            roof = {"bound": "hbm", "kernel": "k_mega_decode (persistent single-launch decode step)",
                    "achieved": token_roof["achieved"], "peak": peak, "unit": "GB/s", "frac": token_roof["frac"],
                    "traffic": ncu_traffic("mega", f"{args.model}/gs{args.group_size}/tp{world}"), "traffic_source": ncu_traffic("source", f"{args.model}/gs{args.group_size}/tp{world}"),
                    "bytes_per_launch": btok, "us_per_launch": tok_ms * 1e3, "peak_source": peak_src}
        if world == 1:
            m.set_decode_path(0)
        for kind in (("gate_up", "down", "qkv", "o_proj", "lm_head") if world == 1 else ()):
            ms, nbytes, n = m.bench_kernel(kind, 0, reps=3 if kind != "lm_head" else 1)
            kernels[kind] = {"us": ms * 1e3, "GBps": nbytes / ms / 1e6, "bytes": nbytes}
        if world == 1 and persistent:
            m.set_decode_path(1)  # back on the path that was timed (parity block below)
        if not persistent:
            g = kernels["gate_up"]
            roof = {"bound": "hbm", "kernel": "gate/up int8 GEMV + SwiGLU (k_gemv<EPI_SWIGLU>)",
                    "achieved": g["GBps"], "peak": peak, "unit": "GB/s", "frac": g["GBps"] / peak,
                    "traffic": ncu_traffic("gate_up", f"{args.model}/gs{args.group_size}/tp{world}"), "bytes_per_launch": g["bytes"], "us_per_launch": g["us"],
                    "peak_source": peak_src}
    except Exception as e:  # noqa: BLE001
        log(f"[bench] kernel roofline failed: {e}")

    # ---- batched prefill (tcgen05 int8 GEMM path), secondary metric of BASELINE.json ----
    prefill = None
    if pms is not None and pms == pms:
        try:
            Tn = min(2048, args.ctx)
            ah, kvd = shape.n_heads * shape.head_dim, shape.n_kv_heads * shape.head_dim
            ops = 2.0 * Tn * shape.n_layers * (2 * shape.dim * ah + 2 * shape.dim * kvd + 3 * shape.dim * shape.hidden_dim)
            prefill = {"tokens": Tn, "ms": pms, "value": Tn / pms * 1e3, "unit": "tok/s", "gemm_int8_TOPS": ops / pms / 1e9,
                       "frac_of_int8_peak_4500_TOPS_spec": ops / pms / 1e9 / 4500.0,
                       "note": "whole prefill (norm/quantize, tcgen05 GEMMs with per-group TMEM drains, tensor-core causal attention on an FP16 hi/lo "
                               "split; under tensor parallelism the row-parallel partial blocks are summed over NVLink peer loads); GEMM TOPS counts "
                               "the int8 MACs only; peak is the datasheet figure (the same tiling as a dense int8 GEMM: profiles/r02_gemm_q8_ceilings.txt)"}
        except Exception as e:  # noqa: BLE001
            log(f"[bench] prefill measurement failed: {e}")
    elif prefill_err:
        log(f"[bench] prefill measurement failed: {prefill_err}")

    cpu, parity = None, None
    if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
        try:
            v, cores, dt, oseq, ologits = cpu_decode_tok_s(path, args.ctx, args.cpu_sample_tokens)
            cpu = {"value": v, "unit": "tok/s", "cores": cores, "kind": "port",
                   "sample": f"{args.cpu_sample_tokens} greedy tokens of the same {args.model} gs{args.group_size} .bin after 1 untimed token ({dt:.1f}s), all host threads"}
            if not args.no_extras:
                parity = parity_block(m, oseq, ologits, args)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] cpu baseline / parity failed: {e}")

    long_ctx = prefill_4b = None
    if world == 1 and not args.no_extras:
        m.close()
        m = None
        try:
            long_ctx = long_context_line(path, args, shape, peak, local_rank)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] long-context line failed: {e}")
        try:
            prefill_4b = prefill_4b_line(args, local_rank)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] 4B prefill line failed: {e}")

    out = {
        "metric": "decode_tokens_per_s", "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None,
        "dtype": "int8 weights x int8 activations, int32 group dots, f32 accumulate", "data": "synthetic",
        "config": workload_config(args), "parallelism": ("tp%d" % world) if world > 1 else "single", "where": "cuda",
        "wall_ms_per_step": wall_ms / args.steps,
        "e2e": {"value": e2e_val, "unit": "tok/s", "h2d_bytes_per_step": 16 * tps, "d2h_bytes_per_step": vocab * 4 * tps,
                "tokens_timed": e2e_tokens, "positions": [pos_start, pos_start + n_tok], "path": "Transformer.forward -> host logits -> host argmax (sampler.rs)"},
        "gpu_launches": launches_per_token * n_tok,
        "launches_per_token": launches_per_token,
        "clocks": clk, "roofline": roof, "token_roofline": token_roof, "graph_path_kernels": kernels, "cpu_baseline": cpu,
        "decode_path": "persistent" if persistent else "graph", "prefill": prefill,
        "parity": parity, "exact_mode_tok_s": (parity or {}).get("exact", {}).get("tok_s"), "long_context": long_ctx, "prefill_4b": prefill_4b,
    }
    emit(out)
    if m is not None:
        m.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
