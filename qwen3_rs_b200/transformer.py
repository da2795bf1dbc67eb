"""Host-side mirror of qwen3-inference's model interface over libqwen3cuda's C ABI.

Same names, argument meaning and error behaviour as the reference (models/mod.rs):

    TransformerBuilder::new(path).with_ctx_length(opt).build() -> Transformers   (:40-74)
    Transformer::forward(token, pos) -> &[f32]                                   (:15)
    Transformer::get_config() -> &ModelConfig                                    (:17)

The forward pass runs only in the CUDA library: there is NO CPU fallback -- if the library or a
GPU is missing, construction raises.  numpy arrays returned by forward() are copies of the
logits (the reference hands out a borrow that generate_next_token copies, generation.rs:159-160).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import build as _build


class Q3Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[q3 error {code}] {msg}")
        self.code = code
        self.message = msg


class _Cfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "architecture_id", "dim", "hidden_dim", "n_layers", "n_heads", "n_kv_heads", "head_dim", "seq_len",
        "vocab_size", "group_size", "shared_classifier")]


@dataclass(frozen=True)
class ModelConfig:
    """configuration.rs:18-30."""
    architecture_id: int
    dim: int
    hidden_dim: int
    n_layers: int
    n_heads: int
    n_kv_heads: int
    head_dim: int
    seq_len: int
    vocab_size: int
    group_size: int
    shared_classifier: bool


_lib = None

# every symbol include/qwen3_cuda.h declares: (restype, argtypes)
_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
_pp = C.POINTER(C.c_void_p)
ABI = {
    "q3_create": (_i, [C.c_char_p, _i, _i, _pp]),
    "q3_create_tp": (_i, [C.c_char_p, _i, _i, _i, _i, _pp]),
    "q3_tp_blob_size": (_sz, []),
    "q3_tp_export": (_i, [_vp, _vp]),
    "q3_tp_connect": (_i, [_vp, _vp]),
    "q3_tp_set_logits_root": (_i, [_vp, _i]),
    "q3_destroy": (None, [_vp]),
    "q3_get_config": (C.POINTER(_Cfg), [_vp]),
    "q3_forward": (_i, [_vp, _i, _i, _vp]),
    "q3_forward_argmax": (_i, [_vp, _i, _i, C.POINTER(_i)]),
    "q3_decode_greedy": (_i, [_vp, _i, _i, _i, _vp]),
    "q3_sampler_set": (_i, [_vp, _f, _f, C.c_ulonglong]),
    "q3_sampler_state": (_i, [_vp, C.POINTER(C.c_ulonglong)]),
    "q3_sampler_skip": (_i, [_vp, _i]),
    "q3_forward_sample": (_i, [_vp, _i, _i, C.POINTER(_i)]),
    "q3_decode_sample": (_i, [_vp, _i, _i, _i, _vp]),
    "q3_prefill": (_i, [_vp, _vp, _i, _i, _vp]),
    "q3_bench_prefill": (_i, [_vp, _vp, _i, _i, C.POINTER(_f)]),
    "q3_score": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "q3_score_topk": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "q3_reset": (_i, [_vp]),
    "q3_logits_device": (_vp, [_vp]),
    "q3_logits_host": (_vp, [_vp]),
    "q3_kv_read": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "q3_kv_write": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "q3_forward_layers": (_i, [_vp, _i, _i, _i, _vp, _i, _vp]),
    "q3_set_decode_path": (_i, [_vp, _i]),
    "q3_set_exact": (_i, [_vp, _i]),
    "q3_set_exact_mask": (_i, [_vp, _i]),
    "q3_bench_decode": (_i, [_vp, _i, _i, _i, C.POINTER(_f)]),
    "q3_bench_kernel": (_i, [_vp, _i, _i, _i, C.POINTER(_f), C.POINTER(_i), C.POINTER(C.c_double)]),
    "q3_debug_profile": (_i, [_vp, _i, _i, _vp, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "q3_num_sms": (_i, [_vp]),
    "q3_debug_set_epoch": (_i, [_vp, C.c_ulonglong]),
    "q3_launches_per_step": (_i, [_vp]),
    "q3_op_quantize": (_i, [_i, _vp, _i, _i, _vp, _vp]),
    "q3_op_matmul": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "q3_op_expf": (_i, [_i, _vp, _i, _vp]),
    "q3_op_gemm_q8": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "q3_op_sample": (_i, [_i, _vp, _i, _f, _f, C.POINTER(C.c_ulonglong), C.POINTER(_i)]),
    "q3_bench_gemm_q8": (_i, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(_f)]),
    "q3_op_prefill_attention": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "q3_op_logprobs": (_i, [_i, _vp, _i, _i, _vp, _vp, _vp]),
    "q3_op_topk_logprobs": (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "q3_op_rmsnorm": (_i, [_i, _vp, _vp, _i, _vp]),
    "q3_op_quantize_q80": (_i, [_i, _vp, _sz, _i, _vp, _vp]),
    "q3_op_quantize_q80_dev": (_i, [_i, _vp, _sz, _i, _vp, _vp]),
    "q3_last_error": (C.c_char_p, []),
    "q3_version": (C.c_char_p, []),
}


def lib_path() -> str:
    return _build.LIB


def load_library():
    """dlopen libqwen3cuda.so (building it first if nvcc is present and it is stale)."""
    global _lib
    if _lib is None:
        path = os.environ.get("Q3_LIB") or _build.LIB  # Q3_LIB: a tuning variant built by scripts/ab_variants.py
        if not os.path.exists(path):
            path = _build.build()
        L = C.CDLL(path)
        for name, (res, args) in ABI.items():
            try:
                fn = getattr(L, name)  # AttributeError == missing export: fail loudly
            except AttributeError:
                if os.environ.get("Q3_LIB"):  # an older kernel-tuning variant timed for comparison: entry points added since are absent
                    continue
                raise
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise Q3Error(rc, load_library().q3_last_error().decode(errors="replace"))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Transformer:
    """Device-resident Qwen3 transformer (the `Transformers::Qwen3` variant, models/mod.rs:20-37)."""

    def __init__(self, handle: int, tp_size: int = 1):
        self._h = handle
        self._tp_size = tp_size
        c = load_library().q3_get_config(handle).contents
        self._config = ModelConfig(**{n: (bool(getattr(c, n)) if n == "shared_classifier" else int(getattr(c, n)))
                                      for n, _ in _Cfg._fields_})
        # the handle's own page-locked logits buffer, wrapped without a copy (q3_logits_host): forward() DMA-s into it
        hp = load_library().q3_logits_host(self._h)
        self._logits = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_float)), shape=(self._config.vocab_size,)) if hp else \
            np.empty(self._config.vocab_size, np.float32)

    # -- the reference trait --------------------------------------------------------------
    def forward(self, token: int, pos: int, copy: bool = True) -> np.ndarray:
        """Transformer::forward.  Out-of-range token/pos raises (the reference panics).  copy=False returns a view of the
        transformer's own logits buffer, valid until the next call -- what the reference's `forward(..) -> &[f32]` hands out."""
        _check(load_library().q3_forward(self._h, int(token), int(pos), _ptr(self._logits)))
        return self._logits.copy() if copy else self._logits

    def get_config(self) -> ModelConfig:
        return self._config

    # -- extensions (SURVEY §8f) ----------------------------------------------------------
    def forward_argmax(self, token: int, pos: int) -> int:
        out = C.c_int(0)
        _check(load_library().q3_forward_argmax(self._h, int(token), int(pos), C.byref(out)))
        return out.value

    def decode_greedy(self, first_token: int, pos0: int, n: int) -> List[int]:
        out = np.zeros(max(n, 1), np.int32)
        _check(load_library().q3_decode_greedy(self._h, int(first_token), int(pos0), int(n), _ptr(out)))
        return out[:n].tolist()

    # -- device sampler (sampler.rs on the device) --------------------------------------------
    def sampler_set(self, temperature: float, topp: float, rng_seed: int) -> None:
        """Sampler::new(vocab_size, temperature, topp, rng_seed) -- state lives on the device."""
        _check(load_library().q3_sampler_set(self._h, float(temperature), float(topp), int(rng_seed) & 0xFFFFFFFFFFFFFFFF))

    @property
    def sampler_rng_state(self) -> int:
        out = C.c_ulonglong(0)
        _check(load_library().q3_sampler_state(self._h, C.byref(out)))
        return out.value

    def sampler_skip(self, n_draws: int) -> None:
        _check(load_library().q3_sampler_skip(self._h, int(n_draws)))

    def forward_sample(self, token: int, pos: int) -> int:
        out = C.c_int(0)
        _check(load_library().q3_forward_sample(self._h, int(token), int(pos), C.byref(out)))
        return out.value

    def decode_sample(self, first_token: int, pos0: int, n: int) -> List[int]:
        out = np.zeros(max(n, 1), np.int32)
        _check(load_library().q3_decode_sample(self._h, int(first_token), int(pos0), int(n), _ptr(out)))
        return out[:n].tolist()

    def prefill(self, tokens: Sequence[int], pos0: int = 0, want_logits: bool = True) -> Optional[np.ndarray]:
        t = np.ascontiguousarray(tokens, np.int32)
        _check(load_library().q3_prefill(self._h, _ptr(t), t.size, int(pos0), _ptr(self._logits) if want_logits else None))
        return self._logits.copy() if want_logits else None

    def bench_prefill(self, tokens: Sequence[int], pos0: int = 0) -> float:
        t = np.ascontiguousarray(tokens, np.int32)
        ms = C.c_float(0)
        _check(load_library().q3_bench_prefill(self._h, _ptr(t), t.size, int(pos0), C.byref(ms)))
        return ms.value

    def score(self, tokens: Sequence[int], targets: Optional[Sequence[int]] = None, pos0: int = 0, want_argmax: bool = True):
        """q3_score: run `tokens` at positions pos0.. in one batched pass -> (logprobs, argmax).  logprobs[i] is the natural-log
        probability of targets[i] after tokens[:i + 1] (None without targets); argmax[i] the greedy token there (None unless
        want_argmax).  Leaves the KV cache as prefill(tokens, pos0) does."""
        t = np.ascontiguousarray(tokens, np.int32).reshape(-1)
        tg = None if targets is None else np.ascontiguousarray(targets, np.int32).reshape(-1)
        if tg is not None and tg.size != t.size:
            raise ValueError(f"score: {tg.size} targets for {t.size} tokens")
        lp = None if tg is None else np.empty(t.size, np.float32)
        am = np.empty(t.size, np.int32) if want_argmax else None
        _check(load_library().q3_score(self._h, _ptr(t), t.size, int(pos0), _ptr(tg), _ptr(lp), _ptr(am)))
        return lp, am

    def score_topk(self, tokens: Sequence[int], k: int, targets: Optional[Sequence[int]] = None, pos0: int = 0,
                   want_argmax: bool = True):
        """q3_score_topk: score() plus the k most likely tokens at every position -> (ids [n, k], lps [n, k], logprobs,
        argmax).  Row i of ids is in descending probability, equal values with the larger id first (ids[:, 0] is the argmax);
        lps holds their natural-log probabilities.  logprobs / argmax as in score() and bit-identical to its results."""
        t = np.ascontiguousarray(tokens, np.int32).reshape(-1)
        tg = None if targets is None else np.ascontiguousarray(targets, np.int32).reshape(-1)
        if tg is not None and tg.size != t.size:
            raise ValueError(f"score_topk: {tg.size} targets for {t.size} tokens")
        k = _topk_k(k)
        ids = np.empty((t.size, k), np.int32)
        lps = np.empty((t.size, k), np.float32)
        lp = None if tg is None else np.empty(t.size, np.float32)
        am = np.empty(t.size, np.int32) if want_argmax else None
        _check(load_library().q3_score_topk(self._h, _ptr(t), t.size, int(pos0), k, _ptr(ids), _ptr(lps), _ptr(tg), _ptr(lp),
                                            _ptr(am)))
        return ids, lps, lp, am

    def reset(self) -> None:
        _check(load_library().q3_reset(self._h))

    def kv_read(self, layer: int, pos0: int, n: int):
        """Rows [pos0, pos0 + n) of one layer's K and V cache.  A tensor-parallel member holds (and returns / takes in
        kv_write) only its own n_kv_heads / tp_size heads."""
        kv = self._config.n_kv_heads // self._tp_size * self._config.head_dim
        k = np.empty((n, kv), np.float32)
        v = np.empty((n, kv), np.float32)
        _check(load_library().q3_kv_read(self._h, layer, pos0, n, _ptr(k), _ptr(v)))
        return k, v

    def kv_write(self, layer: int, pos0: int, k: np.ndarray, v: np.ndarray) -> None:
        k = np.ascontiguousarray(k, np.float32)
        v = np.ascontiguousarray(v, np.float32)
        kv = self._config.n_kv_heads // self._tp_size * self._config.head_dim
        if k.shape != v.shape or k.ndim != 2 or k.shape[1] != kv:
            raise ValueError(f"kv_write expects [n][{kv}] rows (this handle's kv heads)")
        _check(load_library().q3_kv_write(self._h, layer, pos0, k.shape[0], _ptr(k), _ptr(v)))

    def forward_layers(self, x: np.ndarray, pos: int, layer0: int, layer1: int, run_head: bool = False):
        x = np.array(x, np.float32)
        lg = np.empty(self._config.vocab_size, np.float32) if run_head else None
        _check(load_library().q3_forward_layers(self._h, int(pos), layer0, layer1, _ptr(x), int(run_head), _ptr(lg)))
        return (x, lg) if run_head else x

    def set_exact(self, on: bool) -> None:
        """Reference-order reductions + glibc expf: logits bit-identical to the reference (slow)."""
        _check(load_library().q3_set_exact(self._h, int(on)))

    def set_exact_mask(self, mask: int) -> None:
        """Reference order for a subset of the reductions (see q3_set_exact_mask in include/qwen3_cuda.h)."""
        _check(load_library().q3_set_exact_mask(self._h, int(mask)))

    def set_decode_path(self, path: int) -> None:
        _check(load_library().q3_set_decode_path(self._h, path))

    def bench_decode(self, first_token: int, pos0: int, steps: int) -> float:
        ms = C.c_float(0)
        _check(load_library().q3_bench_decode(self._h, first_token, pos0, steps, C.byref(ms)))
        return ms.value

    KERNEL_KINDS = {"qkv": 0, "o_proj": 1, "gate_up": 2, "down": 3, "lm_head": 4, "attention": 5}

    def bench_kernel(self, kind: str, pos: int = 0, reps: int = 4):
        """-> (avg ms per launch, algorithmic bytes per launch, launches)."""
        ms, n, b = C.c_float(0), C.c_int(0), C.c_double(0)
        _check(load_library().q3_bench_kernel(self._h, self.KERNEL_KINDS[kind], pos, reps, C.byref(ms), C.byref(n), C.byref(b)))
        return ms.value / max(n.value, 1), b.value, n.value

    def debug_profile(self, token: int, pos: int) -> np.ndarray:
        """Per-CTA tagged clock stamps of one persistent-kernel decode step: [3 * num_sms, n_events] of (clock64 << 8 | tag),
        rows [0, num_sms) from consumer thread 0, [num_sms, 2 num_sms) from producer 0, [2 num_sms, 3 num_sms) from the
        first lane of consumer group 1 (same SM clock); the last column is the row's event count (prof_mark in
        csrc/q3_mega.cuh).  The buffer is sized from the library's own answer."""
        rows, ev = C.c_int(0), C.c_int(0)
        _check(load_library().q3_debug_profile(self._h, token, pos, None, 0, C.byref(rows), C.byref(ev)))
        buf = np.zeros((rows.value, ev.value), np.uint64)
        _check(load_library().q3_debug_profile(self._h, token, pos, _ptr(buf), buf.size, C.byref(rows), C.byref(ev)))
        return buf

    @property
    def num_sms(self) -> int:
        return load_library().q3_num_sms(self._h)

    def debug_set_epoch(self, exchanges_issued: int) -> None:
        _check(load_library().q3_debug_set_epoch(self._h, int(exchanges_issued)))

    @property
    def launches_per_step(self) -> int:
        return load_library().q3_launches_per_step(self._h)

    # -- tensor parallelism (one process per GPU; see tp_connect below) -------------------------
    def tp_export(self) -> bytes:
        n = load_library().q3_tp_blob_size()
        buf = C.create_string_buffer(n)
        _check(load_library().q3_tp_export(self._h, buf))
        return buf.raw

    def tp_connect_blobs(self, blobs: bytes) -> None:
        _check(load_library().q3_tp_connect(self._h, C.create_string_buffer(blobs, len(blobs))))

    def tp_set_logits_root(self, root: int) -> None:
        _check(load_library().q3_tp_set_logits_root(self._h, int(root)))

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._logits = np.array(self._logits, np.float32)  # detach from the handle's page-locked buffer before it is freed
            load_library().q3_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TransformerBuilder:
    """models/mod.rs:40-74."""

    def __init__(self, checkpoint_path: str):
        self.checkpoint_path = checkpoint_path
        self.ctx_length: Optional[int] = None
        self.device = 0
        self.tp_rank, self.tp_size = 0, 1

    @staticmethod
    def new(checkpoint_path: str) -> "TransformerBuilder":
        return TransformerBuilder(checkpoint_path)

    def with_ctx_length(self, ctx_length: Optional[int]) -> "TransformerBuilder":
        self.ctx_length = ctx_length
        return self

    def with_device(self, device: int) -> "TransformerBuilder":
        self.device = device
        return self

    def with_tensor_parallel(self, rank: int, size: int) -> "TransformerBuilder":
        self.tp_rank, self.tp_size = rank, size
        return self

    def build(self) -> Transformer:
        L = load_library()
        h = C.c_void_p(0)
        ctx = int(self.ctx_length) if self.ctx_length else 0
        if self.tp_size == 1:
            rc = L.q3_create(self.checkpoint_path.encode(), ctx, self.device, C.byref(h))
        else:
            rc = L.q3_create_tp(self.checkpoint_path.encode(), ctx, self.device, self.tp_rank, self.tp_size, C.byref(h))
        _check(rc)
        return Transformer(h.value, self.tp_size)


def tp_connect(m: Transformer, dist) -> None:
    """Exchange the ranks' CUDA-IPC blobs over torch.distributed (plumbing only) and map the peers'
    exchange buffers.  Every rank of the group must call this after build()."""
    import torch

    blob = m.tp_export()
    world = dist.get_world_size()
    if dist.get_backend() == "nccl":
        mine = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
        allb = torch.empty(world * len(blob), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(allb, mine)
        blobs = bytes(allb.cpu().numpy().tobytes())
    else:
        objs = [None] * world
        dist.all_gather_object(objs, blob)
        blobs = b"".join(objs)
    m.tp_connect_blobs(blobs)
    dist.barrier()


# ---- operator-level entry points (tests) ---------------------------------------------------
def op_quantize(x: np.ndarray, gs: int, device: int = 0):
    x = np.ascontiguousarray(x, np.float32)
    q = np.empty(x.size, np.int8)
    s = np.empty(x.size // gs, np.float32)
    _check(load_library().q3_op_quantize(device, _ptr(x), x.size, gs, _ptr(q), _ptr(s)))
    return q, s


def op_expf(x, device: int = 0):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty_like(x)
    _check(load_library().q3_op_expf(device, _ptr(x), x.size, _ptr(out)))
    return out


def op_matmul(xq, xs, wq, ws, n: int, d: int, gs: int, want_dots: bool = False, exact: bool = False, device: int = 0):
    xq = np.ascontiguousarray(xq, np.int8)
    xs = np.ascontiguousarray(xs, np.float32)
    wq = np.ascontiguousarray(wq, np.int8)
    ws = np.ascontiguousarray(ws, np.float32)
    out = np.empty(d, np.float32)
    dots = np.empty((d, n // gs), np.int32) if want_dots else None
    _check(load_library().q3_op_matmul(device, _ptr(xq), _ptr(xs), _ptr(wq), _ptr(ws), n, d, gs, int(exact), _ptr(out), _ptr(dots)))
    return (out, dots) if want_dots else out


def op_gemm_q8(xq, xs, wq, ws, T: int, N: int, K: int, gs: int, exact: bool = False, device: int = 0):
    xq = np.ascontiguousarray(xq, np.int8)
    xs = np.ascontiguousarray(xs, np.float32)
    wq = np.ascontiguousarray(wq, np.int8)
    ws = np.ascontiguousarray(ws, np.float32)
    out = np.empty((T, N), np.float32)
    _check(load_library().q3_op_gemm_q8(device, _ptr(xq), _ptr(xs), _ptr(wq), _ptr(ws), T, N, K, gs, int(exact), _ptr(out)))
    return out


def op_sample(logits, temperature: float, topp: float, rng_state: int, device: int = 0):
    """One Sampler::sample draw on the device -> (token, new rng_state)."""
    a = np.ascontiguousarray(logits, np.float32)
    st, tok = C.c_ulonglong(int(rng_state) & 0xFFFFFFFFFFFFFFFF), C.c_int(0)
    _check(load_library().q3_op_sample(device, _ptr(a), a.size, float(temperature), float(topp), C.byref(st), C.byref(tok)))
    return tok.value, st.value


def op_prefill_attention(q, k, v, pos0: int, n_heads: int, n_kv: int, device: int = 0):
    """Causal attention of T = q.shape[0] query tokens at positions pos0.. over k / v rows [pos0 + T][n_kv * 128], with the
    tensor-core kernel q3_prefill runs (FP16 hi / lo split)."""
    q = np.ascontiguousarray(q, np.float32)
    k = np.ascontiguousarray(k, np.float32)
    v = np.ascontiguousarray(v, np.float32)
    out = np.empty_like(q)
    _check(load_library().q3_op_prefill_attention(device, _ptr(q), _ptr(k), _ptr(v), q.shape[0], pos0, n_heads, n_kv, _ptr(out)))
    return out


def bench_gemm_q8(T: int, N: int, K: int, gs: int = 64, mode: int = 0, reps: int = 5, device: int = 0) -> float:
    """Milliseconds per launch of the tcgen05 GEMM alone (mode 0 fast drain, 1 exact drain)."""
    ms = C.c_float(0)
    _check(load_library().q3_bench_gemm_q8(device, T, N, K, gs, mode, reps, C.byref(ms)))
    return ms.value


def op_logprobs(logits, targets=None, want_argmax: bool = True, device: int = 0):
    """q3_score's reduction on logits [rows][n] -> (log softmax(row)[targets[r]] or None, last argmax of each row or None)."""
    a = np.ascontiguousarray(logits, np.float32)
    a = a.reshape(1, -1) if a.ndim == 1 else a
    rows, n = a.shape
    tg = None if targets is None else np.ascontiguousarray(targets, np.int32).reshape(-1)
    if tg is not None and tg.size != rows:
        raise ValueError(f"op_logprobs: {tg.size} targets for {rows} rows")
    lp = None if tg is None else np.empty(rows, np.float32)
    am = np.empty(rows, np.int32) if want_argmax else None
    _check(load_library().q3_op_logprobs(device, _ptr(a), rows, n, _ptr(tg), _ptr(lp), _ptr(am)))
    return lp, am


TOPK_MAX = 64  # Q3_TOPK_MAX in include/qwen3_cuda.h


def _topk_k(k) -> int:
    if isinstance(k, bool) or int(k) != k or not 1 <= k <= TOPK_MAX:
        raise ValueError(f"k must be an integer in 1 .. {TOPK_MAX}, got {k!r}")
    return int(k)


def op_topk_logprobs(logits, k: int, targets=None, want_argmax: bool = True, device: int = 0):
    """q3_score_topk's reduction on logits [rows][n] -> (ids [rows, k], lps [rows, k], log softmax(row)[targets[r]] or None,
    last argmax of each row or None)."""
    a = np.ascontiguousarray(logits, np.float32)
    a = a.reshape(1, -1) if a.ndim == 1 else a
    rows, n = a.shape
    tg = None if targets is None else np.ascontiguousarray(targets, np.int32).reshape(-1)
    if tg is not None and tg.size != rows:
        raise ValueError(f"op_topk_logprobs: {tg.size} targets for {rows} rows")
    k = _topk_k(k)
    ids = np.empty((rows, k), np.int32)
    lps = np.empty((rows, k), np.float32)
    lp = None if tg is None else np.empty(rows, np.float32)
    am = np.empty(rows, np.int32) if want_argmax else None
    _check(load_library().q3_op_topk_logprobs(device, _ptr(a), rows, n, k, _ptr(tg), _ptr(ids), _ptr(lps), _ptr(lp), _ptr(am)))
    return ids, lps, lp, am


def op_rmsnorm(x, w, device: int = 0):
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w, np.float32)
    out = np.empty_like(x)
    _check(load_library().q3_op_rmsnorm(device, _ptr(x), _ptr(w), x.size, _ptr(out)))
    return out


def op_quantize_q80_dev(w_ptr: int, n: int, gs: int, q_ptr: int, s_ptr: int, device: int = 0) -> None:
    """quantize_q80 on device buffers given as raw device addresses (e.g. torch tensors' data_ptr())."""
    _check(load_library().q3_op_quantize_q80_dev(device, C.c_void_p(w_ptr), n, gs, C.c_void_p(q_ptr), C.c_void_p(s_ptr)))


def op_quantize_q80(w, gs: int, device: int = 0):
    w = np.ascontiguousarray(w, np.float32).reshape(-1)
    q = np.empty(w.size, np.int8)
    s = np.empty(w.size // gs, np.float32)
    _check(load_library().q3_op_quantize_q80(device, _ptr(w), w.size, gs, _ptr(q), _ptr(s)))
    return q, s, None
