"""Regenerates tests/golden/hf_qwen3_logits.npz, Hugging Face's Qwen3 logits that tests/test_oracle_vs_hf.py compares the
oracle with (run from the repo root: python tests/golden/make_hf_golden.py; needs transformers).

For each case of the test: the prompt tokens, HF's fp32 CPU logits of the whole prompt, and the logits of the two negative
controls (RoPE base 1e4 instead of 1e6, RMSNorm epsilon 1e-1).  Stored as float16: that rounding moves the relative
errors the test measures by about 1e-4, against tolerances of a few per cent."""
import os
import sys
import tempfile

import numpy as np
import torch
import transformers

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_oracle_vs_hf import CASES, HF_GOLDEN, prepare  # noqa: E402


def hf_logits(hf_dir, tokens, **override):
    from transformers import AutoConfig, Qwen3ForCausalLM
    cfg = AutoConfig.from_pretrained(hf_dir)
    for k, v in override.items():
        setattr(cfg, k, v)
        if k == "rope_theta" and getattr(cfg, "rope_parameters", None):  # transformers >= 5 keeps the base here
            cfg.rope_parameters = dict(cfg.rope_parameters, rope_theta=v)
    model = Qwen3ForCausalLM.from_pretrained(hf_dir, config=cfg, torch_dtype=torch.float32).eval()
    with torch.no_grad():
        return model(torch.tensor([tokens])).logits[0].numpy()


def main():
    arrays = {}
    for name, gs, seed in CASES:
        with tempfile.TemporaryDirectory() as d:
            hf_dir, _, tokens = prepare(d, name, gs, seed)
            key = f"{name}_gs{gs}_s{seed}"
            arrays[key + "_tokens"] = np.array(tokens, np.int32)
            arrays[key + "_logits"] = hf_logits(hf_dir, tokens).astype(np.float16)
            arrays[key + "_logits_rope_theta_1e4"] = hf_logits(hf_dir, tokens, rope_theta=10000.0).astype(np.float16)
            arrays[key + "_logits_rms_norm_eps_1e-1"] = hf_logits(hf_dir, tokens, rms_norm_eps=1e-1).astype(np.float16)
    np.savez_compressed(HF_GOLDEN, **arrays)
    print(f"wrote {HF_GOLDEN} (transformers {transformers.__version__}, torch {torch.__version__})")


if __name__ == "__main__":
    main()
