"""An independent anchor for the oracle's ARCHITECTURE: Hugging Face's Qwen3 (transformers, fp32, CPU) on the same synthetic
weights.  The reference exports HF checkpoints and claims to compute the same network with int8 weights and int8
activations; its own forward path has no tests, so the oracle (a restatement of the reference) is compared here with the
canonical implementation the checkpoints come from.  Quantisation noise is a few per cent; a wrong convention (RoPE pairing
or base, missing QK-norm, GQA head mapping, norm epsilon placement, SwiGLU order) moves the logits by O(1) - the negative
controls show the test can tell the difference.

HF's logits are stored in tests/golden/hf_qwen3_logits.npz (float16; tests/golden/make_hf_golden.py regenerates them with
transformers), so the comparison does not depend on which transformers release, if any, is installed."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR
from oracle import binding as orc
from qwen3_rs_b200 import export, synth

CASES = [("tiny", 64, 2), ("tiny-untied", 64, 1)]
HF_GOLDEN = os.path.join(GOLDEN_DIR, "hf_qwen3_logits.npz")


def prepare(tmp_dir, name, gs, seed):
    """-> (HF checkpoint directory, the .bin the repo's exporter makes of it, prompt tokens) of one case."""
    shape = synth.SHAPES[name]
    hf_dir = synth.write_hf_dir(shape, os.path.join(tmp_dir, "hf"), seed=seed, dtype="f32")
    cfg = json.load(open(os.path.join(hf_dir, "config.json")))
    cfg.update(model_type="qwen3", rope_theta=1000000.0, hidden_act="silu", attention_bias=False)  # what Qwen3 checkpoints say
    json.dump(cfg, open(os.path.join(hf_dir, "config.json"), "w"))
    out = os.path.join(tmp_dir, "m.bin")
    export.export_model(hf_dir, out, gs)
    rng = np.random.default_rng(seed)
    tokens = rng.integers(0, shape.vocab_size, 24).tolist()
    return hf_dir, out, tokens


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.mark.parametrize("name,gs,seed", CASES)
def test_oracle_agrees_with_hf_qwen3_up_to_quantisation_noise(tmp_path, name, gs, seed):
    _, out, tokens = prepare(str(tmp_path), name, gs, seed)
    hf = np.load(HF_GOLDEN)
    key = f"{name}_gs{gs}_s{seed}"
    assert hf[key + "_tokens"].tolist() == tokens
    want = hf[key + "_logits"].astype(np.float32)          # [T, vocab], causal attention over the whole prompt
    o = orc.Model(out)
    got = np.stack([o.forward(t, p) for p, t in enumerate(tokens)])
    errs = np.array([_rel(got[p], want[p]) for p in range(len(tokens))])
    corr = min(float(np.corrcoef(got[p], want[p])[0, 1]) for p in range(len(tokens)))
    print(f"{name}: oracle vs HF fp32: rel err median {np.median(errs):.3f} max {errs.max():.3f}, min corr {corr:.5f}")
    assert errs.max() < 0.08 and np.median(errs) < 0.05 and corr > 0.995
    # negative controls: the same comparison against an HF model with ONE convention changed must be clearly worse
    wrong_theta = hf[key + "_logits_rope_theta_1e4"].astype(np.float32)
    e_theta = np.array([_rel(got[p], wrong_theta[p]) for p in range(8, len(tokens))])   # positions where the angle differs
    wrong_eps = hf[key + "_logits_rms_norm_eps_1e-1"].astype(np.float32)
    e_eps = np.array([_rel(got[p], wrong_eps[p]) for p in range(len(tokens))])
    print(f"   controls: rope base 1e4 -> median {np.median(e_theta):.3f}; rms eps 1e-1 -> median {np.median(e_eps):.3f}")
    assert np.median(e_theta) > 3 * np.median(errs[8:]) and np.median(e_eps) > 3 * np.median(errs)
