"""Synthetic (random-init, seeded) Qwen3 checkpoints of the BASELINE.json shapes.

Real checkpoints are unavailable offline, so parity tests and the bench run on random weights of
the named architectures (SURVEY.md §8d): an HF-layout directory (config.json + model.safetensors,
tensor names per qwen3-export/src/models/qwen3.rs:12-33) that is then run through the repo's own
exporter (`export.py`).  For the multi-GB shapes `export_synthetic` streams tensor by tensor
straight into the exporter instead of materialising a 16 GB safetensors file first; the
quantizer and the byte layout are the same code either way.

Init (chosen so activations/logits stay O(1) and greedy argmax margins are far above the 1e-2
logit tolerance): linear weights N(0, 1/in_features); embedding N(0, embed_std^2) with
embed_std = 0.25 (an N(0,1) embedding dominates the residual stream and a tied model then just
repeats its input token -- a degenerate greedy sequence); norm weights 1 + N(0, 0.1^2); untied
lm_head N(0, lm_head_gain^2/dim).
"""
from __future__ import annotations

import json
import os
from dataclasses import dataclass, asdict
from typing import Dict, Iterator, Optional, Tuple

import numpy as np
import torch

from .export import (
    EMBED_TOKENS_KEY,
    LAYER_COMPONENTS,
    LM_HEAD_KEY,
    ExportConfig,
    export_from_loader,
    quantize_q80,
)


@dataclass(frozen=True)
class Shape:
    name: str
    dim: int
    hidden_dim: int
    n_layers: int
    n_heads: int
    n_kv_heads: int
    head_dim: int = 128
    vocab_size: int = 151936
    max_seq_len: int = 40960
    tied: bool = True

    def export_config(self) -> ExportConfig:
        return ExportConfig(self.dim, self.hidden_dim, self.n_layers, self.n_heads, self.n_kv_heads,
                            self.vocab_size, self.max_seq_len, self.head_dim)

    @property
    def weight_elems(self) -> int:
        """int8 elements streamed per decoded token (SURVEY.md §8 table)."""
        ah, kv = self.n_heads * self.head_dim, self.n_kv_heads * self.head_dim
        return self.n_layers * (2 * self.dim * ah + 2 * self.dim * kv + 3 * self.dim * self.hidden_dim) \
            + self.vocab_size * self.dim

    def bytes_per_token(self, group_size: int, pos: int = 0) -> float:
        """Algorithmic bytes per decoded token: W(1+4/gs) + f32 KV read of pos+1 rows (§8d)."""
        kv = self.n_kv_heads * self.head_dim
        return self.weight_elems * (1.0 + 4.0 / group_size) + 2.0 * self.n_layers * (pos + 1) * kv * 4


SHAPES: Dict[str, Shape] = {
    # real Qwen3 architectures (HF configs)
    "qwen3-0.6b": Shape("qwen3-0.6b", 1024, 3072, 28, 16, 8, tied=True),
    "qwen3-1.7b": Shape("qwen3-1.7b", 2048, 6144, 28, 16, 8, tied=True),
    "qwen3-4b": Shape("qwen3-4b", 2560, 9728, 36, 32, 8, tied=True),
    "qwen3-8b": Shape("qwen3-8b", 4096, 12288, 36, 32, 8, tied=False),
    # small test shapes (same op graph; sized so the CPU oracle runs in milliseconds)
    "tiny": Shape("tiny", 256, 768, 2, 4, 2, vocab_size=1024, max_seq_len=256, tied=True),
    "tiny-untied": Shape("tiny-untied", 256, 512, 3, 8, 2, vocab_size=768, max_seq_len=128, tied=False),
    "small": Shape("small", 512, 1536, 4, 8, 4, vocab_size=4096, max_seq_len=512, tied=True),
    "micro": Shape("micro", 128, 384, 2, 2, 1, vocab_size=256, max_seq_len=64, tied=False),
    "small8": Shape("small8", 512, 2048, 3, 16, 8, vocab_size=4096, max_seq_len=256, tied=False),  # 8 kv heads: tensor parallel up to 8
    # wider than 4096 like Qwen3-32B (5120): the dim > 4096 prefill norm kernel, and the graph decode path as the default (the
    # persistent kernel declines this width); GQA 8, n_heads * 128 == dim; at T 640 every prefill GEMM has more tiles than SMs
    "wide": Shape("wide", 5120, 3072, 2, 40, 5, vocab_size=4096, max_seq_len=2048, tied=False),
}


def hf_config_dict(shape: Shape) -> dict:
    """Fields read by config_loader.rs:128-146."""
    return {
        "architectures": ["Qwen3ForCausalLM"],
        "hidden_size": shape.dim,
        "intermediate_size": shape.hidden_dim,
        "num_hidden_layers": shape.n_layers,
        "num_attention_heads": shape.n_heads,
        "num_key_value_heads": shape.n_kv_heads,
        "vocab_size": shape.vocab_size,
        "max_position_embeddings": shape.max_seq_len,
        "rms_norm_eps": 1e-6,
        "head_dim": shape.head_dim,
        "bos_token_id": 151643,
        "eos_token_id": 151645,
        "tie_word_embeddings": shape.tied,
    }


def tensor_specs(shape: Shape) -> Iterator[Tuple[str, Tuple[int, ...], str]]:
    """(name, shape, kind) for every tensor of the HF checkpoint, kind in norm|embed|linear|head."""
    ah, kv = shape.n_heads * shape.head_dim, shape.n_kv_heads * shape.head_dim
    out_in = {
        "self_attn.q_proj": (ah, shape.dim), "self_attn.k_proj": (kv, shape.dim),
        "self_attn.v_proj": (kv, shape.dim), "self_attn.o_proj": (shape.dim, ah),
        "mlp.gate_proj": (shape.hidden_dim, shape.dim), "mlp.down_proj": (shape.dim, shape.hidden_dim),
        "mlp.up_proj": (shape.hidden_dim, shape.dim),
    }
    yield EMBED_TOKENS_KEY, (shape.vocab_size, shape.dim), "embed"
    for i in range(shape.n_layers):
        yield f"model.layers.{i}.input_layernorm.weight", (shape.dim,), "norm"
        yield f"model.layers.{i}.post_attention_layernorm.weight", (shape.dim,), "norm"
        yield f"model.layers.{i}.self_attn.q_norm.weight", (shape.head_dim,), "norm"
        yield f"model.layers.{i}.self_attn.k_norm.weight", (shape.head_dim,), "norm"
        for comp in LAYER_COMPONENTS:
            yield f"model.layers.{i}.{comp}.weight", out_in[comp], "linear"
    yield "model.norm.weight", (shape.dim,), "norm"
    if not shape.tied:
        yield LM_HEAD_KEY, (shape.vocab_size, shape.dim), "head"


def _name_seed(seed: int, name: str) -> int:
    h = 1469598103934665603
    for b in name.encode():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return (h ^ (seed * 0x9E3779B97F4A7C15)) & 0x7FFFFFFFFFFFFFFF


def make_tensor(name: str, tshape: Tuple[int, ...], kind: str, seed: int, lm_head_gain: float = 4.0,
                device: str = "cpu", bf16_round: bool = True, embed_std: float = 0.25) -> torch.Tensor:
    """One tensor, f32, a pure function of (seed, name) so any subset can be regenerated.
    Values are rounded through bf16 (what an HF checkpoint stores) when bf16_round."""
    g = torch.Generator(device=device)
    g.manual_seed(_name_seed(seed, name))
    t = torch.randn(tshape, generator=g, device=device, dtype=torch.float32)
    if kind == "norm":
        t = 1.0 + 0.1 * t
    elif kind == "linear":
        t = t * (1.0 / float(tshape[1]) ** 0.5)
    elif kind == "embed":
        t = t * embed_std
    elif kind == "head":
        t = t * (lm_head_gain / float(tshape[1]) ** 0.5)
    if bf16_round:
        t = t.to(torch.bfloat16).to(torch.float32)
    return t


def write_hf_dir(shape: Shape, out_dir: str, seed: int = 0, dtype: str = "bf16") -> str:
    """config.json + model.safetensors (BF16 or F32 -- both are read by tensor_reader.rs:92-106)."""
    from safetensors.torch import save_file

    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "config.json"), "w") as f:
        json.dump(hf_config_dict(shape), f, indent=1)
    tensors = {}
    for name, tshape, kind in tensor_specs(shape):
        t = make_tensor(name, tshape, kind, seed)
        tensors[name] = t.to(torch.bfloat16) if dtype == "bf16" else t
    save_file(tensors, os.path.join(out_dir, "model.safetensors"))
    return out_dir


def quantize_q80_device(t: torch.Tensor, group_size: int):
    """export.quantize_q80 evaluated by the library's own device quantiser (k_quantize_q80 behind
    q3_op_quantize_q80_dev: IEEE division + round-half-to-even, bit-identical to the numpy exporter -- tested in
    tests/test_gpu_parity.py); `t` is a CUDA tensor.  Used to make the multi-GB bench / test checkpoints quickly."""
    from . import transformer as T

    w = t.reshape(-1).contiguous()
    q = torch.empty(w.numel(), dtype=torch.int8, device=w.device)
    s = torch.empty(w.numel() // group_size, dtype=torch.float32, device=w.device)
    torch.cuda.synchronize(w.device)
    T.op_quantize_q80_dev(w.data_ptr(), w.numel(), group_size, q.data_ptr(), s.data_ptr(), w.device.index or 0)
    return q.cpu().numpy(), s.cpu().numpy(), 0.0


def export_synthetic(shape: Shape, output_path: str, group_size: int = 64, seed: int = 0,
                     device: str = "cpu", quantizer=None) -> dict:
    """Stream make_tensor() -> exporter without the intermediate safetensors file.  Produces the
    same bytes as write_hf_dir(dtype='bf16') + export_model() (tested on the small shapes)."""
    specs = {name: (tshape, kind) for name, tshape, kind in tensor_specs(shape)}

    def load(name: str):
        if name not in specs:
            return None
        tshape, kind = specs[name]
        t = make_tensor(name, tshape, kind, seed, device=device)
        # quantised tensors may stay on the device for a device-side quantizer; norms are written as f32
        return t if (quantizer is not None and device != "cpu" and kind != "norm") else t.cpu().numpy()

    info = export_from_loader(load, shape.export_config(), output_path, group_size,
                              shared_classifier=shape.tied, quantizer=quantizer or quantize_q80)
    info.update(shape=asdict(shape), seed=seed)
    return info


def checkpoint_bytes(shape: Shape, group_size: int) -> int:
    """Size of the exported .bin (SURVEY.md appendix A)."""
    # embed doubles as lm_head when tied (stored once); otherwise embed + separate lm_head
    n_q = shape.weight_elems + (0 if shape.tied else shape.vocab_size * shape.dim)
    norms = (2 * shape.n_layers * shape.dim + shape.dim + 2 * shape.n_layers * shape.head_dim) * 4
    return 256 + norms + n_q + (n_q // group_size) * 4
